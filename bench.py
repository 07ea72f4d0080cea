#!/usr/bin/env python
"""Benchmark of the SoW training hot path on B200 (contract: see the task's bench.py section).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): SoW Llama-350M r=50 bf16 pre-training tokens/s (reference definition, simple_train.py:
609,680-690: global non-pad tokens per optimizer update / time per update), synthetic tokens, random-init weights.
One "step" = one optimizer update of the training loop (forward, backward, gradient averaging, fused AdamW) in
steady state (after >= 1 merge, dense W present).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama_350m",
                    help="llama_{9m,60m,130m,350m,7b} (pre-training / keep fine-tune) or roberta_base (BASELINE.json configs[2]: "
                         "GLUE-shaped fine-tune, mode keep, rank 8, seq 512, batch 16 -- pass those flags)")
    ap.add_argument("--rank", type=int, default=50)
    ap.add_argument("--batch", type=int, default=128,
                    help="sequences per GPU per step (128 = the reference's documented pre-training recipe, readme.md:5-26)")
    ap.add_argument("--seq", type=int, default=256)
    ap.add_argument("--mode", default="pretrain", choices=["pretrain", "keep"],
                    help="pretrain: empty accumulation, everything trains (config 2); keep: fine-tune of a dense model, "
                         "frozen base, only the factors train (configs 3-4)")
    ap.add_argument("--act-ckpt", action="store_true", help="activation checkpointing (config 4: Llama-7B)")
    ap.add_argument("--param-dtype", default="bf16", choices=["bf16", "f32"],
                    help="dtype of the model parameters (the reference's GLUE scripts never set one: fp32)")
    ap.add_argument("--compile", action="store_true",
                    help="torch.compile(model) around the custom-op SoW layers (scripts/finetune.py:486-487); the reference-on-GPU "
                         "baseline is compiled too.  Secondary row: the headline is the eager run")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="replay forward+backward+optimizer as ONE CUDA graph (single GPU; for small per-GPU batches, which are "
                         "launch-bound).  Use --warmup >= 5: the capture happens on the 4th step after a merge")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-rows", action="store_true", help="skip the batch-16/64 and torch.compile rows")
    ap.add_argument("--no-fused-optimizer", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32): its loss and "
                         "every parameter after the optimizer update, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_BYTES = 60_000_000          # float32 data; with the .npy headers a dump stays under 64 MB


def dump_outputs(out_dir, loss, model):
    """The results of the last timed step as float32 .npy files: the loss it returned and the parameters its optimizer
    update left behind.  A parameter larger than its share of DUMP_BYTES is sampled at positions drawn from a fixed seed.
    The inputs (weights, token batches) are seeded too, so two builds run with the same arguments can be compared output
    for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    params = [(n, p) for n, p in model.named_parameters() if p.numel()]
    per_param = DUMP_BYTES // 4 // (len(params) + 1)
    gen = torch.Generator().manual_seed(0)
    for name, p in params:
        flat = p.detach().reshape(-1)
        if flat.numel() > per_param:
            flat = flat[torch.randint(flat.numel(), (per_param,), generator=gen).to(flat.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), flat.float().cpu().numpy())


def load_traffic():
    """ncu-measured DRAM bytes per launch of the kernels the roofline names, with the profiles/ file they come from."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


SHAPES = {   # scripts/configs/*.json of the reference (data): hidden, intermediate, layers
    "llama_9m": (128, 352, 4), "llama_60m": (512, 1376, 8), "llama_130m": (768, 2048, 12),
    "llama_350m": (1024, 2736, 24), "llama_7b": (4096, 11008, 32), "roberta_base": (768, 3072, 12),
}


def workload_name(args):
    h, ff, L = SHAPES[args.model]
    if args.model.startswith("roberta"):
        kind = "GLUE-shaped fine-tuning (sequence classification, synthetic labels, mode keep, frozen base)"
    elif args.mode == "pretrain":
        kind = "pre-training"
    else:
        kind = "fine-tuning (mode keep, frozen base" + (", activation checkpointing" if args.act_ckpt else "") + ")"
    return (f"{args.model} (h={h}, ff={ff}, L={L}) SoW rank {args.rank} {kind}, seq {args.seq}, steady state after 1 merge "
            f"(dense W), fwd+bwd+grad-avg+AdamW per step")


def run_ref_subprocess(extra, timeout=1500):
    """Run baseline/ref_runner.py (the unmodified reference from baseline/_ref, own interpreter because its package is
    also called tn_gradient) and return its JSON line, or None when baseline/_ref is absent or the run failed."""
    runner = os.path.join(ROOT, "baseline", "ref_runner.py")
    if not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "tn_gradient", "layer", "sow.py")):
        return None
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        res = subprocess.run([sys.executable, runner] + [str(a) for a in extra], capture_output=True, text=True,
                             timeout=timeout, env=env, cwd=os.path.join(ROOT, "baseline"))
    except Exception:
        return None
    for ln in reversed(res.stdout.strip().splitlines()):
        if ln.startswith("{"):
            try:
                return json.loads(ln)
            except ValueError:
                pass
    sys.stderr.write("[bench] reference runner failed:\n" + res.stderr[-2000:] + "\n")
    return None


def ref_workload_args(args):
    """Same workload for the reference arm as for ours (model, rank, seq, mode, scale, optimizer hyper-parameters)."""
    if args.model.startswith("roberta"):
        return ["--model", args.model, "--rank", args.rank, "--seq", args.seq, "--mode", "keep", "--scale", 1.0,
                "--lr", 5e-5, "--sow-lr", 1.2e-4]
    return ["--model", args.model, "--rank", args.rank, "--seq", args.seq, "--mode", args.mode,
            "--scale", 1.0 if args.mode == "pretrain" else 0.125]


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, all host threads.
    Drives the UNMODIFIED reference package (baseline/_ref: stock tn_gradient.prepare.prepare_sow / SoWLinear /
    accumulate, installed by baseline/install_ref.sh) in the loop order of scripts/simple_train.py:596-650; falls
    back to the oracle port (oracle/cpu_trainer.py) only when baseline/_ref is absent.  Each step is a bounded
    sample of the workload (2 sequences instead of the per-GPU batch) so that the run ends within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_batch = 2
    t0 = time.time()
    W = max(1, args.warmup)
    res = run_ref_subprocess(ref_workload_args(args) + ["--batch", sample_batch, "--steps", args.steps, "--warmup", W,
                                                        "--device", "cpu", "--dtype", "f32", "--merge-at", 0])
    kind = "reference"
    if res is None:
        from oracle.cpu_trainer import time_cpu_training
        res = time_cpu_training(args.model, args.rank, batch=sample_batch, seq_len=args.seq, steps=args.steps, warmup=W)
        kind = "port"
    line = {
        "impl": "reference", "metric": "train_tokens_per_s", "value": res["tokens_per_s"], "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": W,
        "ms_per_step": res["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "sample": f"{sample_batch} x {args.seq} tokens per step on host cores (fp32, the reference's stock "
                             f"SoWLinear / prepare_sow / accumulate from baseline/_ref)" if kind == "reference" else
                             f"{sample_batch} x {args.seq} tokens per step on host cores (fp32, oracle port)"},
        "cpu_baseline": {"value": res["tokens_per_s"], "unit": "tokens/s", "cores": res["threads"], "kind": kind,
                         "sample": f"{args.steps} steps of {sample_batch}x{args.seq} tokens, merge in warm-up"},
        "e2e": {"value": res["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from sow_b200 import ops
    from sow_b200.trainer import SoWTrainer, TrainConfig

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    peaks = load_peaks()

    roberta = args.model.startswith("roberta")
    if roberta:
        args.mode = "keep"
        # run_glue.py recipe (readme.md:30-67): lr 5e-5, sow_lr 1.2e-4, scale 1 until the first merge, then 1/rank
        cfg = TrainConfig(model=args.model, rank=args.rank, seq_len=args.seq, batch_size=args.batch, lr=5e-5, sow_lr=1.2e-4,
                          fused_optimizer=not args.no_fused_optimizer, decompose="keep", freeze_base=True,
                          activation_checkpointing=args.act_ckpt, scale=1.0, scale_after_first_merge=1.0 / args.rank,
                          dtype=torch.float32 if args.param_dtype == "f32" else torch.bfloat16)
    else:
        cfg = TrainConfig(model=args.model, rank=args.rank, seq_len=args.seq, batch_size=args.batch,
                          fused_optimizer=not args.no_fused_optimizer, decompose="keep" if args.mode == "keep" else None,
                          freeze_base=args.mode == "keep", activation_checkpointing=args.act_ckpt,
                          scale=1.0 if args.mode == "pretrain" else 0.125,
                          dtype=torch.float32 if args.param_dtype == "f32" else torch.bfloat16)
    cfg.compile = bool(args.compile)
    cfg.cuda_graph = bool(args.cuda_graph)
    trainer = SoWTrainer(cfg, device)
    B, S = args.batch, args.seq
    n_batches = 8
    gen = torch.Generator().manual_seed(1234 + rank)                      # SURVEY.md 8d: per-rank stream
    if roberta:
        host_batches = [torch.randint(3, 50265, (B, S), generator=gen, dtype=torch.int64).pin_memory() for _ in range(n_batches)]
        host_labels = [torch.randint(0, 2, (B,), generator=gen, dtype=torch.int64).pin_memory() for _ in range(n_batches)]
    else:
        host_batches = [torch.randint(1, 32000, (B, S), generator=gen, dtype=torch.int64).pin_memory() for _ in range(n_batches)]
        host_labels = [None] * n_batches
    dev_batches = [b.to(device) for b in host_batches]
    dev_labels = [None if l is None else l.to(device) for l in host_labels]
    _step = trainer.step

    class _T:          # trainer.step with the labels of the batch (sequence classification) or labels = input_ids (causal LM)
        @staticmethod
        def step(ids, i=None):
            lab = None
            if roberta:
                lab = dev_labels[i % n_batches] if i is not None else dev_labels[0]
            return _step(ids, labels=lab)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: W steps, the first followed by a merge so that the timed steps see a dense W --------------
    W = max(args.warmup, 3)
    for i in range(W):
        loss = _T.step(dev_batches[i % n_batches], i)
        if i == 0:
            trainer.merge()
    barrier()

    # ---- timed region 1: inputs resident in HBM --------------------------------------------------------------
    K = args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_counter["kernels"]
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loss = _T.step(dev_batches[i % n_batches], i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_counter["kernels"] - launches0
    clocks = sampler.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms)
    tokens_per_step = B * S * world
    value = tokens_per_step * K / (ms_max / 1e3)
    final_loss = float(loss)
    if args.dump_outputs and rank == 0:                  # replicas hold identical parameters
        dump_outputs(args.dump_outputs, loss, trainer.model)

    # ---- timed region 2: end to end through the public API with HOST buffers -------------------------------
    barrier()
    e0.record()
    for i in range(K):
        ids = host_batches[i % n_batches].to(device, non_blocking=True)   # H2D of this step's inputs (pinned)
        lab = host_labels[i % n_batches].to(device, non_blocking=True) if roberta else None
        loss = trainer.step(ids, labels=lab)
        _ = loss.item()                                                    # D2H of the step's result
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = tokens_per_step * K / (float(ms2) / 1e3)

    # ---- instrumented pass: CUDA events around every kernel of each class (not part of `value`) -------------
    trainer.cfg.cuda_graph = False           # the per-launch events need real launches, not a graph replay
    trainer.invalidate_graph()
    ops.profile_enable(True)
    for i in range(args.profile_steps):
        _T.step(dev_batches[i % n_batches], i)
    torch.cuda.synchronize()
    kern = {}
    for k in ops.PROF_CLASSES:
        tms, work, n = ops.profile_read(k)
        kern[k] = {"ms_total": tms, "work": work, "launches": n}
    ops.profile_enable(False)
    # merge events, each timed by CUDA events inside the C ABI around the single grouped launch.  As in training
    # (simple_train.py:618-626) the merge is issued right behind a backward pass, with no host synchronisation in
    # between, so the GPU is at its working clocks.  After the first merge B = 0, so repeated merges leave W unchanged
    # numerically while moving exactly the same bytes.
    merge_ms, merge_event_ms, merge_event_wall_ms = [], [], []
    mg_bytes = 0.0
    for i in range(5):
        torch.cuda.synchronize()
        ops.profile_enable(True)
        _T.step(dev_batches[i % n_batches], i)
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw = time.perf_counter()
        m0.record()
        trainer.merge()               # accumulate(model) + reset_optimizer: merge kernel, thin-QR re-init, broadcast of A_new
        m1.record()
        torch.cuda.synchronize()
        merge_event_wall_ms.append((time.perf_counter() - tw) * 1e3)
        merge_event_ms.append(m0.elapsed_time(m1))
        ms_i, mg_bytes, mg_n = ops.profile_read("merge")
        ops.profile_enable(False)
        merge_ms.append(ms_i)
    mg_ms = statistics.median(merge_ms)

    # TT-Adam on a Llama-7B-shaped bf16 weight (BASELINE.json config 5), order 2: fused update + re-compression
    tt_rows = {}
    if rank == 0:
        from tn_gradient.optimizer.ttadam import TTAdam
        for r_tt in (8, 64):
            Mt = Nt = 4096
            p_tt = torch.nn.Parameter((torch.randn(Mt, Nt, device=device) * 0.02).to(torch.bfloat16))
            p_tt.grad = (torch.randn(Mt, Nt, device=device) * 0.01).to(torch.bfloat16)
            opt_tt = TTAdam([{"params": [p_tt], "ranks": [1, r_tt, 1]}], lr=1e-3)
            for _ in range(3):
                opt_tt.step()
            torch.cuda.synchronize()
            # ten optimizer steps issued back to back (as in training: no host synchronisation between parameters)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(10):
                opt_tt.step()
            a1.record()
            torch.cuda.synchronize()
            t_ms = a0.elapsed_time(a1) / 10
            # algorithmic bytes (SURVEY.md 8d): fused Adam g + p r/w = 6 B/elem; two decompositions 4*P*P each + cores
            P_tt = 64 * 64
            fused_bytes = Mt * Nt * 6
            survey_bytes = fused_bytes + 2 * 4 * P_tt * P_tt + 2 * 4 * P_tt * P_tt + 4 * 4 * r_tt * 2 * P_tt
            tt_rows[f"ttadam_4096x4096_order2_r{r_tt}"] = {
                "bound": "hbm", "ms_per_step": t_ms, "unit": "GB/s", "peak": peaks["hbm_gbs"],
                "achieved_fused_accounting": fused_bytes / t_ms / 1e6, "frac_fused_accounting": fused_bytes / t_ms / 1e6 / peaks["hbm_gbs"],
                "achieved_survey_accounting": survey_bytes / t_ms / 1e6, "frac_survey_accounting": survey_bytes / t_ms / 1e6 / peaks["hbm_gbs"],
                "note": "fused: bytes this implementation must move (g, p r/w); survey: + dense fp32 moments written and "
                        "re-read by two decompositions (SURVEY.md 8d formula for an unfused pipeline)"}
            del opt_tt, p_tt
        # the same update over EIGHT independent parameters in one optimizer step (a model's step): TTAdam alternates them between
        # side streams, so one parameter's QR chain overlaps another's main kernel
        for r_tt in (8, 64):
            Mt = Nt = 4096
            ps_tt = [torch.nn.Parameter((torch.randn(Mt, Nt, device=device) * 0.02).to(torch.bfloat16)) for _ in range(8)]
            for p_tt in ps_tt:
                p_tt.grad = (torch.randn(Mt, Nt, device=device) * 0.01).to(torch.bfloat16)
            opt_tt = TTAdam([{"params": ps_tt, "ranks": [1, r_tt, 1]}], lr=1e-3)
            for _ in range(3):
                opt_tt.step()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(5):
                opt_tt.step()
            a1.record()
            torch.cuda.synchronize()
            t_ms = a0.elapsed_time(a1) / 5 / len(ps_tt)
            fused_bytes = Mt * Nt * 6
            tt_rows[f"ttadam_8x4096x4096_order2_r{r_tt}"] = {
                "bound": "hbm", "ms_per_parameter": t_ms, "unit": "GB/s", "peak": peaks["hbm_gbs"],
                "achieved_fused_accounting": fused_bytes / t_ms / 1e6,
                "frac_fused_accounting": fused_bytes / t_ms / 1e6 / peaks["hbm_gbs"],
                "note": "eight independent parameters per optimizer step, tensor-train updates alternating between side streams"}
            del opt_tt, ps_tt
        torch.cuda.empty_cache()

    # dominant kernel: the fused SoW GEMM (forward y and backward dX are the same kernel template)
    gemm_ms = kern["gemm_fwd"]["ms_total"] + kern["gemm_dx"]["ms_total"]
    gemm_flops = kern["gemm_fwd"]["work"] + kern["gemm_dx"]["work"]
    gemm_n = kern["gemm_fwd"]["launches"] + kern["gemm_dx"]["launches"]
    achieved_tf = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    peak_tf = peaks["bf16_tflops_sustained"]
    step_ms = ms_max / K
    traffic = load_traffic()
    roofline = {
        "kernel": "sow_gemm_kernel<BN=256> (y_i = x.W_i + t_i.B_i and the group dX = sum_i dY_i.W_i^T + dt_cat.A_cat^T, "
                  "tcgen05/TMEM/TMA)",
        "bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
        "frac": achieved_tf / peak_tf if peak_tf else None,
        "frac_of_burst_peak": achieved_tf / peaks["bf16_tflops"] if peaks["bf16_tflops"] else None,
        "flops_accounting": "algorithmic, un-padded rank (SURVEY.md 8d)",
        # dram__bytes_read + dram__bytes_write of ONE forward launch at the bench shape, from the committed ncu --set full
        # capture named in profiles/r02_traffic.json (null until that capture exists for this shape)
        "traffic": traffic.get("gemm_fwd", {}).get("bytes") if B * S == traffic.get("gemm_fwd", {}).get("T") else None,
        "traffic_source": traffic.get("gemm_fwd", {}).get("source"),
        "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
        "launches_timed": gemm_n, "avg_launch_us": 1e3 * gemm_ms / max(gemm_n, 1),
        "share_of_step": (gemm_ms / max(args.profile_steps, 1)) / step_ms,
        "share_of_step_fwd": (kern["gemm_fwd"]["ms_total"] / max(args.profile_steps, 1)) / step_ms,
        "share_of_step_dx": (kern["gemm_dx"]["ms_total"] / max(args.profile_steps, 1)) / step_ms,
    }
    merge_gbs = mg_bytes / (mg_ms / 1e3) / 1e9 if mg_ms > 0 else 0.0
    extra_kernels = {
        "merge": {"bound": "hbm", "achieved": merge_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                  "frac": merge_gbs / peaks["hbm_gbs"], "ms": mg_ms, "algorithmic_bytes": mg_bytes, "launches": mg_n,
                  "events": len(merge_ms), "ms_all": merge_ms,
                  # whole merge EVENT as the training loop sees it (simple_train.py:618-626): grouped merge kernel + thin-QR
                  # re-initialisation of every A + zeroing of B + broadcast of A_new + reset_optimizer; CUDA events / host wall
                  "merge_event_ms": statistics.median(merge_event_ms),
                  "merge_event_wall_ms": statistics.median(merge_event_wall_ms),
                  "traffic": traffic.get("merge", {}).get("bytes") if abs(mg_bytes - traffic.get("merge", {}).get("algorithmic_bytes", -1)) < 1 else None,
                  "traffic_source": traffic.get("merge", {}).get("source")},
    }
    extra_kernels.update(tt_rows)
    for k in ("gemm_skinny", "gemm_splitk", "gemm_k2", "adam"):
        d = kern[k]
        if d["ms_total"] > 0:
            rate = d["work"] / (d["ms_total"] / 1e3)
            extra_kernels[k] = {"ms_per_step": d["ms_total"] / args.profile_steps, "launches_per_step": d["launches"] / args.profile_steps,
                                "achieved": rate / (1e9 if k == "adam" else 1e12), "unit": "GB/s" if k == "adam" else "TFLOP/s"}
    side = sum(kern[k]["ms_total"] for k in ("gemm_skinny", "gemm_splitk", "gemm_k2")) / args.profile_steps
    extra_kernels["rank_r_side_path_ms_per_step"] = side          # t_cat + dA_cat + fused dt/dB (round 1: 16.7 ms + pack/finalize)
    fam_ms = gemm_ms + sum(kern[k]["ms_total"] for k in ("gemm_skinny", "gemm_splitk", "gemm_k2"))
    fam_fl = gemm_flops + sum(kern[k]["work"] for k in ("gemm_skinny", "gemm_splitk", "gemm_k2"))
    extra_kernels["sow_gemm_family"] = {"achieved": fam_fl / (fam_ms / 1e3) / 1e12 if fam_ms > 0 else 0.0, "unit": "TFLOP/s",
                                        "frac_of_sustained": fam_fl / (fam_ms / 1e3) / 1e12 / peak_tf if fam_ms > 0 else None,
                                        "ms_per_step": fam_ms / args.profile_steps}
    extra_kernels["gemm_fwd_ms_per_step"] = kern["gemm_fwd"]["ms_total"] / args.profile_steps
    extra_kernels["gemm_dx_ms_per_step"] = kern["gemm_dx"]["ms_total"] / args.profile_steps

    # ---- multi-GPU correctness (world > 1): replicas must hold identical parameters after the timed steps, and identical
    # merged W / re-initialised A after one more merge (SURVEY.md 8e; raises on a mismatch)
    replicas, comm = None, None
    if world > 1:
        # how much of the gradient all-reduce is NOT hidden behind backward: CUDA events on the compute stream around the
        # wait for the bucket all-reduces, 5 steps
        trainer.comm_events = []
        for i in range(5):
            _T.step(dev_batches[i % n_batches], i)
        torch.cuda.synchronize()
        waits = [a.elapsed_time(b) for a, b in trainer.comm_events]
        trainer.comm_events = None
        w_ms = torch.tensor([statistics.median(waits)], device=device, dtype=torch.float64)
        dist.all_reduce(w_ms, op=dist.ReduceOp.MAX)
        comm = {"exposed_allreduce_wait_ms": float(w_ms), "of_step_ms": step_ms,
                "buckets_bytes": [int(b["flat"].numel() * b["flat"].element_size()) for b in trainer.grad_sync.buckets],
                "note": "max over ranks of the median device-side wait between the end of backward and the completion of the last "
                        "bucket all-reduce (NCCL AVG, one call per flat bucket, launched from post-accumulate-grad hooks as the "
                        "bucket fills); the last bucket holds embed_tokens, whose gradient is produced by the very last backward "
                        "kernel, so its all-reduce cannot overlap anything"}
        from sow_b200.parallel import assert_replicas_consistent
        from sow_b200.surgery import sow_modules
        assert_replicas_consistent(list(trainer.model.parameters()), "parameter after the timed steps")
        _T.step(dev_batches[0], 0)
        trainer.merge()
        mods = sow_modules(trainer.model)
        assert_replicas_consistent([m.acc_downweight for m in mods], "merged W")
        assert_replicas_consistent([a for m in mods for a in m.downscale_weights], "re-initialised A")
        replicas = {"consistent": True, "checked": "all parameters after the timed steps; merged W and re-initialised A of "
                    f"{len(mods)} SoW layers after one more merge (bit-exact across {world} ranks)"}

    # ---- BASELINE.json config 2 sweeps the per-GPU batch {16, 64, 128}: small batches are launch-bound (~5 k launches per
    # step), so they are reported eager AND replayed as one CUDA graph (rank 0, N=1 only; not part of `value`)
    def quick_run(batch, graph=False, compiled=False, steps=12, warm=6):
        import copy
        c2 = copy.copy(cfg)
        c2.batch_size, c2.cuda_graph, c2.compile = batch, graph, compiled
        t2 = SoWTrainer(c2, device)
        g2 = torch.Generator().manual_seed(99)
        ids2 = [torch.randint(1, 32000, (batch, S), generator=g2, dtype=torch.int64).to(device) for _ in range(4)]
        for i in range(warm):
            t2.step(ids2[i % 4])
            if i == 0:
                t2.merge()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(steps):
            l2 = t2.step(ids2[i % 4])
        a1.record()
        torch.cuda.synchronize()
        ms2_ = a0.elapsed_time(a1) / steps
        out = {"tokens_per_s": batch * S / (ms2_ / 1e3), "ms_per_step": ms2_, "loss": float(l2)}
        del t2
        torch.cuda.empty_cache()
        return out

    sweep, compiled_row = None, None
    if rank == 0 and world == 1 and not roberta and not args.no_extra_rows and args.model == "llama_350m" and args.mode == "pretrain":
        del trainer
        trainer = None
        torch.cuda.empty_cache()
        sweep = {}
        for b_ in (16, 64):
            sweep[f"batch_{b_}"] = {"eager": quick_run(b_), "cuda_graph": quick_run(b_, graph=True)}
        if not args.compile:
            # torch.compile(model) as scripts/finetune.py:486-487: the SoW layers are registered custom ops (zero graph
            # breaks), inductor fuses the stock HF element-wise code around them
            compiled_row = quick_run(B, compiled=True, steps=8, warm=4)
            compiled_row["what"] = "same step with torch.compile(model); SoW layers traced as sow_b200::linear_fwd/bwd custom ops"

    # ---- CPU baseline (rank 0, N=1 only): the reference's CPU path on the host cores -- the UNMODIFIED reference from
    # baseline/_ref when it is there (kind "reference"), else the oracle port ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = run_ref_subprocess(ref_workload_args(args) + ["--batch", 2, "--steps", 3, "--warmup", 1, "--device", "cpu",
                                                            "--dtype", "f32", "--merge-at", 0])
        kind = "reference"
        if res is None and not roberta:
            from oracle.cpu_trainer import time_cpu_training
            res = time_cpu_training(args.model, args.rank, batch=2, seq_len=S, steps=3, warmup=1)
            kind = "port"
        if res is not None:
            cpu_baseline = {"value": res["tokens_per_s"], "unit": "tokens/s", "cores": res["threads"], "kind": kind,
                            "sample": f"3 steps of 2x{S} tokens ({args.model} SoW r={args.rank}, fp32, merge in warm-up), "
                                      f"{res['sec_per_step']:.2f} s/step"}

    # ---- the reference itself on the SAME GPU at the SAME config (rank 0, N=1 only): stock tn_gradient.SoWLinear /
    # prepare_sow / accumulate from baseline/_ref, eager cuBLAS + torch.optim.AdamW, in its own process -- the practical
    # bar of BASELINE.md section 5, reported beside the CPU baseline, not part of `value`
    gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        trainer = None
        torch.cuda.empty_cache()
        pd = "f32" if args.param_dtype == "f32" else "bf16"
        res = run_ref_subprocess(ref_workload_args(args) + ["--batch", B, "--steps", 5, "--warmup", 3, "--device", "cuda",
                                                            "--dtype", pd, "--merge-at", 0] + (["--compile"] if args.compile else []))
        kind = f"reference (unmodified package from baseline/_ref, eager torch ops, {pd}, torch.optim.AdamW) on the same B200"
        if res is None and not roberta:
            from oracle.cpu_trainer import time_cpu_training
            res = time_cpu_training(args.model, args.rank, batch=B, seq_len=S, steps=5, warmup=3, device=str(device),
                                    dtype=torch.bfloat16)
            kind = "port (eager torch ops of the reference, bf16, torch.optim.AdamW) on the same B200"
        if res is not None:
            gpu_eager = {"value": res["tokens_per_s"], "unit": "tokens/s", "kind": kind, "same_config": True,
                         "sample": f"5 steps of {B}x{S} tokens, {res['sec_per_step'] * 1e3:.1f} ms/step",
                         "speedup_of_this_build": value / res["tokens_per_s"]}
        if compiled_row is not None:
            resc = run_ref_subprocess(ref_workload_args(args) + ["--batch", B, "--steps", 5, "--warmup", 3, "--device", "cuda",
                                                                 "--dtype", pd, "--merge-at", 0, "--compile"])
            if resc is not None:
                compiled_row["reference_compiled_tokens_per_s"] = resc["tokens_per_s"]
                compiled_row["speedup_over_compiled_reference"] = compiled_row["tokens_per_s"] / resc["tokens_per_s"]

    if rank == 0:
        line = {
            "metric": "train_tokens_per_s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.param_dtype == "bf16" else "f32 parameters, bf16x3 tensor-core products", "data": "synthetic",
            "config": {
                "workload": workload_name(args),
                "per_gpu_batch": B, "global_batch": B * world, "seq_len": S, "tokens_per_step": tokens_per_step,
                "parallelism": f"dp{world}", "l2": "working set per step (>1 GB weights+activations) exceeds the 126 MB L2; no flush needed",
                "optimizer": "FusedAdamW (sow_adam_multi)" if cfg.fused_optimizer else "torch.optim.AdamW",
                "torch_compile": bool(args.compile), "cuda_graph": bool(args.cuda_graph),
            },
            "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": B * S * 8 + (B * 8 if roberta else 0),
                    "d2h_bytes_per_step": 4},
            "gpu_launches": launches,
            "roofline": roofline,
            "kernels": extra_kernels,
            "cpu_baseline": cpu_baseline,
            "gpu_eager_baseline": gpu_eager,
            "replicas": replicas,
            "comm": comm,
            "batch_sweep": sweep,
            "compiled": compiled_row,
            "clocks": clocks,
            "loss": final_loss,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
