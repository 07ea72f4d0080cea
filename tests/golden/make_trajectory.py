"""Golden LOSS TRAJECTORY of the unmodified reference (antoine311200/sow at /root/reference): a tiny Llama (the shape
of scripts/configs/llama_*.json scaled down: h=64, ff=176, 2 layers, 4 heads, vocab 512) through the loop of
scripts/simple_train.py:596-650 -- prepare_sow over the 7 projections, AdamW with the two param groups, 6 optimizer
steps with sow_accumulation = 2 (accumulate + reset_optimizer after the backward of steps 3 and 5:
simple_train.py:618-626 merges when update_step > 0 and update_step % sow_accumulation == 0), fp32 on CPU.

Run in the build container only:   cd tests/golden && python make_trajectory.py   -> trajectory.npz
Stores the reference's initial state (so the GPU test starts from identical weights), the token batches, the loss of
every step, and the weights of the first merge.  Nothing of the reference's source is copied.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import import_reference, npy  # noqa: E402

TARGETS = ["q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"]
TINY = dict(hidden_size=64, intermediate_size=176, num_hidden_layers=2, num_attention_heads=4)
VOCAB, SEQ, BATCH, RANK, STEPS, SOW_ACC = 512, 32, 8, 8, 6, 2


def build_tiny():
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=VOCAB, max_position_embeddings=64, rms_norm_eps=1e-6, hidden_act="silu",
                      initializer_range=0.02, bos_token_id=0, eos_token_id=1, use_cache=False, tie_word_embeddings=False,
                      **TINY)
    torch.manual_seed(42)
    return LlamaForCausalLM(cfg)


def reset_optimizer(optimizer, group_id):          # scripts/utils/training_utils.py:257-277
    for p in optimizer.param_groups[group_id]["params"]:
        st = optimizer.state[p]
        if not st:
            continue
        st["exp_avg"] = torch.zeros_like(p)
        st["exp_avg_sq"] = torch.zeros_like(p)
        if "step" in st:
            st["step"] = torch.zeros_like(st["step"])


def main():
    ref_sow, ref_prepare, *_ = import_reference()
    torch.set_num_threads(1)
    model = build_tiny()
    cfg = ref_prepare.SoWConfig(target_modules=TARGETS, rank=RANK, scale=1.0, device="cpu", init_method="normal",
                                decompose=None)
    model = ref_prepare.prepare_sow(model, cfg)
    out = {}
    for k, v in model.state_dict().items():
        out[f"init/{k}"] = npy(v)
    sow = [m for m in model.modules() if isinstance(m, ref_sow.SoWLinear)]
    special = [p for m in sow for p in list(m.downscale_weights) + list(m.upscale_weights)]
    ids = {id(p) for p in special}
    others = [p for p in model.parameters() if p.requires_grad and id(p) not in ids]
    opt = torch.optim.AdamW([{"params": others, "lr": 1e-3, "weight_decay": 0.0},
                             {"params": special, "lr": 1e-3, "weight_decay": 0.0}])
    g = torch.Generator().manual_seed(7)
    losses, batches, merges = [], [], 0
    for step in range(1, STEPS + 1):
        ids_ = torch.randint(1, VOCAB, (BATCH, SEQ), generator=g)
        batches.append(ids_.numpy())
        loss = model(input_ids=ids_, labels=ids_).loss
        loss.backward()
        update_step = step - 1
        if update_step > 0 and update_step % SOW_ACC == 0:       # simple_train.py:618-626: after backward, before the step
            ref_prepare.accumulate(model)
            reset_optimizer(opt, 1)
            merges += 1
            # later merges add A_new.B with a freshly drawn A_new: only the first merged W can be compared
            for name, m in model.named_modules():
                if merges == 1 and isinstance(m, ref_sow.SoWLinear):
                    out[f"merged{step}/{name}.acc_downweight"] = npy(m.acc_downweight)
        opt.step()
        opt.zero_grad()
        losses.append(float(loss.detach()))
    out["losses"] = np.array(losses, dtype=np.float64)
    out["batches"] = np.stack(batches)
    out["meta"] = np.array([VOCAB, SEQ, BATCH, RANK, STEPS, SOW_ACC, TINY["hidden_size"], TINY["intermediate_size"],
                            TINY["num_hidden_layers"], TINY["num_attention_heads"]], dtype=np.int32)
    path = os.path.join(HERE, "trajectory.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path) / 1024:.1f} KiB; losses = {losses}")


if __name__ == "__main__":
    main()
