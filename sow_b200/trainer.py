"""Synthetic-token SoW pre-training harness: the loop of scripts/simple_train.py:596-650 around the kernel-backed
``tn_gradient`` API, without the data / W&B / checkpoint plumbing (SURVEY.md 2, row 7: the driver is the caller
contract, not part of the hot path).

Loop order is the reference's, including its quirk: at a merge step the gradients were computed w.r.t. the OLD
factors, then ``accumulate`` + ``reset_optimizer`` run, then the optimizer applies those gradients to the
re-initialised factors (simple_train.py:618-626 then :646).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn as nn

from .optim import FusedAdamW
from .parallel import FlatGradSync, broadcast_parameters
from .surgery import SoWConfig, accumulate, prepare_sow, sow_modules

# shapes of scripts/configs/*.json in the reference (data, not code); vocab 32000, rms_norm_eps 1e-6, silu
LLAMA_SHAPES: Dict[str, Dict[str, int]] = {
    "llama_9m": dict(hidden_size=128, intermediate_size=352, num_hidden_layers=4, num_attention_heads=4),
    "llama_60m": dict(hidden_size=512, intermediate_size=1376, num_hidden_layers=8, num_attention_heads=8),
    "llama_130m": dict(hidden_size=768, intermediate_size=2048, num_hidden_layers=12, num_attention_heads=12),
    "llama_350m": dict(hidden_size=1024, intermediate_size=2736, num_hidden_layers=24, num_attention_heads=16),
    "llama_7b": dict(hidden_size=4096, intermediate_size=11008, num_hidden_layers=32, num_attention_heads=32),
}
LLAMA_TARGETS = ["q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"]   # simple_train.py:318
ROBERTA_TARGETS = ["query", "key", "value", "output.dense", "intermediate.dense"]               # run_glue.py:572
# scripts/configs/roberta.json (RoBERTa-base): data, not code
ROBERTA_SHAPES: Dict[str, Dict[str, int]] = {
    "roberta_base": dict(hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12),
    "roberta_tiny": dict(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4),
}


def build_llama(name: str, seq_len: int = 256, vocab_size: int = 32000, seed: int = 42,
                dtype: Optional[torch.dtype] = None) -> nn.Module:
    """Random-init HF Llama of the named reference config (AutoModelForCausalLM.from_config, simple_train.py:313-314).
    ``dtype`` builds the parameters directly in that dtype (halves the host memory of the 7B config)."""
    from transformers import LlamaConfig, LlamaForCausalLM
    shp = LLAMA_SHAPES[name]
    cfg = LlamaConfig(vocab_size=vocab_size, max_position_embeddings=max(1024, seq_len), rms_norm_eps=1e-6,
                      hidden_act="silu", initializer_range=0.02, bos_token_id=0, eos_token_id=1, use_cache=False,
                      tie_word_embeddings=False, **shp)
    torch.manual_seed(seed)
    if dtype is None:
        return LlamaForCausalLM(cfg)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        return LlamaForCausalLM(cfg)
    finally:
        torch.set_default_dtype(prev)


def build_roberta(name: str = "roberta_base", seq_len: int = 512, num_labels: int = 2, seed: int = 42,
                  dropout: float = 0.1) -> nn.Module:
    """Random-init HF RoBERTa sequence classifier of the reference's GLUE config (run_glue.py:508-516 loads
    AutoModelForSequenceClassification; no checkpoint is reachable offline, so the weights are random-init)."""
    from transformers import RobertaConfig, RobertaForSequenceClassification
    cfg = RobertaConfig(vocab_size=50265, hidden_act="gelu", hidden_dropout_prob=dropout, attention_probs_dropout_prob=dropout,
                        max_position_embeddings=max(514, seq_len + 2), type_vocab_size=1, layer_norm_eps=1e-5, pad_token_id=1,
                        bos_token_id=0, eos_token_id=2, num_labels=num_labels, **ROBERTA_SHAPES[name])
    torch.manual_seed(seed)
    return RobertaForSequenceClassification(cfg)


def reset_optimizer(optimizer: torch.optim.Optimizer, group_id: int) -> None:
    """Zero the Adam state of one param group after a merge, by REBINDING the state tensors -- the contract of
    scripts/utils/training_utils.py:257-277 that any optimizer used with SoW has to survive."""
    group = optimizer.param_groups[group_id]
    for param in group["params"]:
        state = optimizer.state[param]
        if not state:
            continue
        state["exp_avg"] = torch.zeros_like(param, memory_format=torch.preserve_format)
        state["exp_avg_sq"] = torch.zeros_like(param, memory_format=torch.preserve_format)
        if group.get("amsgrad", False):
            state["max_exp_avg_sq"] = torch.zeros_like(param, memory_format=torch.preserve_format)
        if "step" in state:
            state["step"] = torch.zeros_like(state["step"])


@dataclass
class TrainConfig:
    model: str = "llama_350m"
    rank: int = 50
    seq_len: int = 256
    batch_size: int = 16                 # per GPU
    lr: float = 1e-2                     # readme.md:5-26
    sow_lr: float = 1e-3
    weight_decay: float = 0.0
    sow_accumulation: int = 5000
    gradient_accumulation: int = 1
    grad_clipping: float = 0.0
    init_method: str = "normal_QR"
    scale: float = 1.0
    dtype: torch.dtype = torch.bfloat16
    seed: int = 42
    activation_checkpointing: bool = False
    fused_optimizer: bool = True
    overlap_grad_sync: bool = True
    decompose: Optional[str] = None      # None: pre-training (empty accumulation); "keep": fine-tuning of a dense model
    freeze_base: bool = False            # fine-tuning: only the SoW factors train (run_glue.py:515-516,547-553)
    scale_after_first_merge: Optional[float] = None   # run_glue.py:996-1001 sets module.scale = 1/rank after the first merge
    dropout: float = 0.1                 # RoBERTa only (scripts/configs/roberta.json)
    compile: bool = False                # torch.compile(model) as scripts/finetune.py:486-487 does (SoW layers = custom ops)
    cuda_graph: bool = False             # capture forward + backward + optimizer step in one CUDA graph and replay it
                                         # (small per-GPU batches are launch-bound: ~5 k launches per step); single GPU
    optimizer_state_dtype: Optional[torch.dtype] = None   # FusedAdamW moments: None = parameter dtype, or torch.float32
    loss_scaling: bool = False           # dynamic loss scaling (torch.amp.GradScaler) for fp16 training; capturable optimizer
    loss_scale_init: float = 2.0 ** 16
    loss_scale_growth_interval: int = 2000
    fused_grad_clipping: bool = False    # grad_clipping inside FusedAdamW (device norm: works with loss scaling and cuda_graph)


class SoWTrainer:
    """One process per GPU.  ``step(input_ids)`` = one micro-step of simple_train.py's loop body."""

    def __init__(self, cfg: TrainConfig, device: torch.device, model: Optional[nn.Module] = None,
                 targets: Optional[list] = None):
        """``model``: an already built (and possibly already SoW-prepared) module to train instead of the named config;
        ``targets``: its SoW target module names."""
        if cfg.loss_scaling and not cfg.fused_optimizer:
            raise ValueError("loss_scaling needs the fused optimizer (GradScaler cannot unscale fp16 gradients for "
                             "torch.optim.AdamW)")
        if cfg.loss_scaling and cfg.dtype == torch.bfloat16:
            raise ValueError("loss_scaling is not available for bf16 models: torch.amp.GradScaler has no bf16 inf / nan "
                             "check, and bf16 has fp32's exponent range, so its gradients need no scaling")
        if cfg.fused_grad_clipping and not cfg.fused_optimizer:
            raise ValueError("fused_grad_clipping needs the fused optimizer (the norm is computed inside FusedAdamW.step)")
        if cfg.loss_scaling and cfg.grad_clipping != 0.0 and not cfg.fused_grad_clipping:
            raise ValueError("loss_scaling with grad_clipping is not supported (the norm of scaled fp16 gradients "
                             "overflows)")
        self.cfg = cfg
        self.device = device
        self.is_classifier = cfg.model.startswith("roberta")
        if model is None:
            if self.is_classifier:
                model = build_roberta(cfg.model, cfg.seq_len, seed=cfg.seed, dropout=cfg.dropout)
                targets = targets or ROBERTA_TARGETS
            else:
                big = LLAMA_SHAPES[cfg.model]["hidden_size"] >= 2048
                model = build_llama(cfg.model, cfg.seq_len, seed=cfg.seed, dtype=cfg.dtype if big else None)
                targets = targets or LLAMA_TARGETS
        from .layer import SoWLinear
        if not any(isinstance(m, SoWLinear) for m in model.modules()):
            if cfg.freeze_base and self.is_classifier:
                for p in model.roberta.parameters():                               # run_glue.py:515-516
                    p.requires_grad = False
            sow_cfg = SoWConfig(target_modules=targets or LLAMA_TARGETS, rank=cfg.rank, init_method=cfg.init_method,
                                scale=cfg.scale, decompose=cfg.decompose, device=str(device))
            model = prepare_sow(model, sow_cfg)                                    # simple_train.py:318-331
        special, ids = [], set()
        for m in sow_modules(model):                                                # simple_train.py:389-405
            for p in list(m.downscale_weights) + list(m.upscale_weights):
                special.append(p)
                ids.add(id(p))
        if cfg.activation_checkpointing:
            model.gradient_checkpointing_enable()
            if cfg.freeze_base and hasattr(model, "enable_input_require_grads"):
                model.enable_input_require_grads()       # frozen embeddings: keep the checkpointed segments differentiable
        model = model.to(device=device, dtype=cfg.dtype)                           # simple_train.py:425-428
        if cfg.freeze_base and not self.is_classifier:
            for p in model.parameters():
                if id(p) not in ids:
                    p.requires_grad_(False)
        for p in special:
            p.requires_grad_(True)
        self.trainable = [p for p in model.parameters() if p.requires_grad and id(p) not in ids]
        self.special = special
        self.model = model
        groups = []
        if self.trainable:
            groups.append({"params": self.trainable, "lr": cfg.lr, "weight_decay": cfg.weight_decay})
            if cfg.fused_grad_clipping and cfg.grad_clipping != 0.0:
                groups[-1]["max_grad_norm"] = cfg.grad_clipping       # the set clip_grad_norm_ clips (:631); not the factors
        self.sow_group_id = len(groups)
        groups.append({"params": self.special, "lr": cfg.sow_lr, "weight_decay": cfg.weight_decay})
        if cfg.cuda_graph and not cfg.fused_optimizer:
            raise ValueError("cuda_graph needs the fused optimizer (device-side step counter)")
        self.optimizer = (FusedAdamW(groups, capturable=cfg.cuda_graph or cfg.loss_scaling,
                                     state_dtype=cfg.optimizer_state_dtype) if cfg.fused_optimizer
                          else torch.optim.AdamW(groups))                                               # :502-506
        # loss scaling: found_inf is computed inside scaler.step, after the bucket all-reduce, so every rank skips alike;
        # the capturable optimizer unscales and skips on the device (no host sync, so the step can be graphed)
        self.scaler = (torch.amp.GradScaler(device.type, init_scale=cfg.loss_scale_init,
                                            growth_interval=cfg.loss_scale_growth_interval)
                       if cfg.loss_scaling else None)
        broadcast_parameters(model)                                                # DDP ctor semantics (:566-572)
        self.grad_sync = FlatGradSync(self.trainable + self.special, overlap=cfg.overlap_grad_sync, direct=self.special)
        self.global_step = 0
        self.update_step = 0
        self.merges = 0
        self.forward_fn = torch.compile(self.model) if cfg.compile else self.model
        self._graph = None               # (CUDAGraph, static input_ids, static labels or None, static loss)
        self._graph_warm = 0             # eager steps since the last (in)validation
        self.graph_launches = 0
        self.comm_events = None          # list of (event, event) pairs when the exposed all-reduce time is being measured
        if cfg.cuda_graph and self.grad_sync.world > 1:
            raise ValueError("cuda_graph is implemented for single-GPU steps (the bucket all-reduces are not captured)")

    # ---- CUDA-graph replay of the whole micro-step ------------------------------------------------------------
    def _graph_ok(self, attention_mask) -> bool:
        cfg = self.cfg
        if not cfg.cuda_graph or attention_mask is not None or cfg.gradient_accumulation != 1:
            return False
        if cfg.grad_clipping != 0.0 and not cfg.fused_grad_clipping:
            return False
        nxt = self.update_step                 # a merge fires inside step() when this is a multiple of sow_accumulation
        return not (nxt > 0 and nxt % int(cfg.sow_accumulation) == 0)

    def _graphed_step(self, input_ids, labels):
        """Two eager steps after every (in)validation settle the addresses the graph will bake in (optimizer state, the
        fused optimizer's pointer tables, workspaces, TMA descriptors); then one capture, then replays.  Gradient
        buckets, in-place merges and the pointer-stable workspaces were laid out for exactly this."""
        if self._graph is not None and (self._graph[1].shape != input_ids.shape or
                                        (self._graph[2] is None) != (labels is None)):
            self._graph = None
            self._graph_warm = 0
        if self._graph is None:
            if self._graph_warm < 2:
                self._graph_warm += 1
                return None
            static_ids = input_ids.clone()
            static_lab = None if labels is None else labels.clone()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            from . import ops
            n0 = ops.launch_counter["kernels"]
            with torch.cuda.graph(g):
                loss = self._eager_body(static_ids, static_lab, None)
            self.graph_launches = ops.launch_counter["kernels"] - n0      # sow_b200 kernels inside one replay
            self._graph = (g, static_ids, static_lab, loss)
        g, static_ids, static_lab, loss = self._graph
        static_ids.copy_(input_ids, non_blocking=True)
        if static_lab is not None:
            static_lab.copy_(labels, non_blocking=True)
        g.replay()
        from . import ops
        ops.launch_counter["kernels"] += self.graph_launches
        self.global_step += 1
        self.update_step += 1
        return loss

    def invalidate_graph(self) -> None:
        self._graph = None
        self._graph_warm = 0

    def step(self, input_ids: torch.Tensor, labels: Optional[torch.Tensor] = None,
             attention_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if self._graph_ok(attention_mask):
            out = self._graphed_step(input_ids, labels)
            if out is not None:
                return out
        self.global_step += 1
        loss = self._eager_body(input_ids, labels, attention_mask)
        return loss

    def _eager_body(self, input_ids, labels, attention_mask):
        cfg = self.cfg
        if labels is None:
            labels = input_ids
        kw = {} if attention_mask is None else {"attention_mask": attention_mask}
        loss = self.forward_fn(input_ids=input_ids, labels=labels, **kw).loss      # simple_train.py:611 / run_glue.py:978
        if self.scaler is not None:
            self.scaler.scale(loss / cfg.gradient_accumulation).backward()
        else:
            (loss / cfg.gradient_accumulation).backward()                          # :612-613 (+ overlapped all-reduce)
        accumulation_step = int(cfg.gradient_accumulation * cfg.sow_accumulation)
        G = cfg.gradient_accumulation
        capturing = torch.cuda.is_current_stream_capturing()
        if (not capturing and (self.global_step % G or G == 1) and self.update_step > 0
                and self.update_step % accumulation_step == 0):                    # :618-626
            self.merge()
        if self.comm_events is not None and not capturing:
            # device-side measurement of the EXPOSED part of the gradient all-reduce: the compute stream reaches e0 when
            # backward is done and e1 when every bucket's all-reduce has finished (bench.py, world > 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.grad_sync.synchronize()
            e1.record()
            self.comm_events.append((e0, e1))
        else:
            self.grad_sync.synchronize()      # DDP semantics: gradients are averaged on every micro-step (no no_sync)
        if self.global_step % G != 0:                                              # :628
            return loss.detach()
        if cfg.grad_clipping != 0.0 and not cfg.fused_grad_clipping:
            torch.nn.utils.clip_grad_norm_(self.trainable, cfg.grad_clipping)      # :631
        # fused_grad_clipping: the trainable group's norm and clip run inside optimizer.step, on the averaged gradients
        # (after grad_sync.synchronize above), so every rank computes the same coefficient
        if self.scaler is not None:
            self.scaler.step(self.optimizer)   # a skipped step (inf / nan gradients) still counts as an update step
            self.scaler.update()
        else:
            self.optimizer.step()                                                  # :646
        self.grad_sync.zero_grad()                                                 # :647 (one memset per bucket)
        if not capturing:
            self.update_step += 1
        return loss.detach()

    def merge(self) -> None:
        accumulate(self.model)
        reset_optimizer(self.optimizer, group_id=self.sow_group_id)
        self.merges += 1
        self.invalidate_graph()                # W / optimizer-state addresses may have changed
        if self.merges == 1 and self.cfg.scale_after_first_merge is not None:      # run_glue.py:996-1001
            for m in sow_modules(self.model):
                m.scale = self.cfg.scale_after_first_merge

    def tokens_per_step(self) -> int:
        return self.cfg.batch_size * self.cfg.seq_len
