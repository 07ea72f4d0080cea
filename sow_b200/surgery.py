"""Model surgery and the merge driver -- host-side mirror of ``tn_gradient.prepare`` (reference file
tn_gradient/prepare.py).

``prepare_sow`` swaps matching ``nn.Linear`` modules for kernel-backed ``SoWLinear`` layers, ``accumulate`` merges
every SoW layer of a model in ONE grouped launch (the reference loops layer by layer, prepare.py:219-222).
"""
from __future__ import annotations

import os
from typing import Iterable, List, Optional

import torch
import torch.nn as nn

from .layer import SharedInputGroup, SoWArgs, SoWLinear, accumulate_modules
from .llama_glue import install_llama_glue

try:  # peft is optional: only the base classes are used by the reference (prepare.py:13)
    from peft import PeftConfig as _PeftConfigBase, PeftModel as _PeftModelBase  # type: ignore
except Exception:  # pragma: no cover - peft is not installed in the build image
    class _PeftConfigBase:  # minimal stand-in storing kwargs
        def __init__(self, **kwargs):
            for k, v in kwargs.items():
                setattr(self, k, v)

    class _PeftModelBase(nn.Module):
        pass


class SoWConfig(_PeftConfigBase):
    """Same fields as tn_gradient.prepare.SoWConfig (prepare.py:27-38)."""

    def __init__(self, target_modules, rank=16, scale=1.0, device="cpu", init_method="normal_QR", decompose="keep",
                 fuse_shared_input=True, **kwargs):
        super().__init__(**kwargs)
        self.fuse_shared_input = fuse_shared_input     # extension: group q/k/v and gate/up (group_shared_inputs)
        self.rank = rank
        self.scale = scale
        self.target_modules = target_modules
        self.device = device
        self.init_method = init_method
        self.decompose = decompose
        self.peft_type = "LORA"


def _matches(name: str, module: nn.Module, targets: Iterable[str], max_split: int) -> bool:
    """Suffix match of dotted module names against target_modules (prepare.py:74-83)."""
    if not isinstance(module, nn.Linear):
        return False
    parts = name.split(".")
    if len(parts) == 1 and parts[0] in targets:
        return True
    for i in range(1, min(max_split + 1, len(parts))):
        if ".".join(parts[-i:]) in targets:
            return True
    return False


def prepare_sow(model: nn.Module, config=None, decompose=None, args: Optional[SoWArgs] = None, **kw):
    """Replace target ``nn.Linear`` modules by ``SoWLinear`` (prepare.py:41-179).

    Accepts both call forms found in the reference's scripts:
      * ``prepare_sow(model, SoWConfig(...))``                      scripts/simple_train.py:331, finetune.py:308
      * ``prepare_sow(model, target_modules, decompose=, args=)``    scripts/run_glue.py:574 (legacy SoWArgs form)

    decompose: None -> empty accumulation (pre-training); 'keep' -> W = weight^T copy; 'qr' -> QR split of the
    pretrained weight into a frozen major part and trainable minor factors.
    """
    if not isinstance(config, SoWConfig):
        a = args if args is not None else SoWArgs()
        config = SoWConfig(target_modules=list(config), rank=a.rank, scale=a.scale,
                           device=a.device if a.device is not None else "cpu", init_method=a.init_method,
                           decompose=decompose if decompose is not None else "qr")
    targets = list(config.target_modules)
    max_split = max(len(t.split(".")) for t in targets)
    selected = [(n, m) for n, m in model.named_modules() if _matches(n, m, targets, max_split)]
    modules = dict(model.named_modules())

    for name, module in selected:
        wdtype = module.weight.data.dtype
        layer = SoWLinear(
            in_features=module.in_features, out_features=module.out_features, rank=config.rank, n_iter=1,
            scale=config.scale, init_method=config.init_method, bias=module.bias is not None, dtype=wdtype,
            device=config.device, init_params=config.decompose != "qr",
        )
        layer.virtual_rank = min(module.in_features, module.out_features)   # merges are always dense (prepare.py:120)

        if config.decompose == "qr":
            # one-off host-side step (SURVEY.md 2b: "host PyTorch"): full QR of the pretrained W^T
            keep = config.rank
            qdev = torch.device("cuda") if torch.cuda.is_available() else module.weight.device
            Q, R = torch.linalg.qr(module.weight.data.T.to(qdev, torch.float32))
            W = (Q[:, :-keep] @ R[:-keep, :]).to(wdtype)
            layer.downscale_weights.from_weights([Q[:, -keep:].to(config.device, wdtype).contiguous()])
            layer.upscale_weights.from_weights([R[-keep:, :].to(config.device, wdtype).contiguous()])
            layer.acc_downweight = nn.Parameter(W.to(config.device).contiguous(), requires_grad=False)
        elif config.decompose == "keep":
            layer.acc_downweight = nn.Parameter(module.weight.data.T.to(config.device).contiguous(), requires_grad=False)

        if module.bias is not None:
            layer.bias = module.bias                                   # the original Parameter is reused (prepare.py:155-156)

        if "." in name:
            parent, child = name.rsplit(".", 1)
            setattr(modules[parent], child, layer)
        else:
            setattr(model, name, layer)
        module.weight = None
    if getattr(config, "fuse_shared_input", True):
        group_shared_inputs(model)
    # rotary embedding and SwiGLU of HF Llama blocks as native kernels (bit-identical to the eager chains)
    install_llama_glue(model)
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
    return model


# sibling projections that HF blocks call with the same hidden-state tensor (LlamaAttention / LlamaMLP,
# RobertaSelfAttention): simple_train.py:318 and run_glue.py:572 list them as separate target modules
SHARED_INPUT_SETS = (("q_proj", "k_proj", "v_proj"), ("gate_proj", "up_proj"), ("query", "key", "value"))


def group_shared_inputs(model: nn.Module, name_sets=SHARED_INPUT_SETS) -> int:
    """Tie sibling SoW projections that read the same input into a SharedInputGroup (SURVEY.md 8f-4): one pass over x
    for all their rank-r down-projections and factor gradients, one dX launch.  Purely an execution plan: parameters,
    state-dict keys and call sites are unchanged, and a group verifies at run time that its members really receive the
    identical tensor (otherwise it switches itself off).  Returns the number of groups formed."""
    formed = 0
    for parent in model.modules():
        kids = dict(parent.named_children())
        for names in name_sets:
            members = [kids[n] for n in names if isinstance(kids.get(n), SoWLinear)]
            if len(members) < 2 or len({m.in_features for m in members}) != 1:
                continue
            grp = SharedInputGroup(members)
            for i, m in enumerate(members):
                m._group = grp
                m._group_index = i
            formed += 1
    return formed


class SoWModel(_PeftModelBase):
    """Thin holder mirroring tn_gradient.prepare.SoWModel (prepare.py:181-185)."""

    def __init__(self, model, config: SoWConfig):
        nn.Module.__init__(self)
        self.config = config
        self.model = prepare_sow(model, config)

    def forward(self, *a, **k):
        return self.model(*a, **k)


def sow_modules(model: nn.Module) -> List[SoWLinear]:
    return [m for _, m in model.named_modules() if isinstance(m, SoWLinear)]


def accumulate(model: nn.Module, sync_reinit: bool = True) -> None:
    """Merge + re-initialise every SoW layer (prepare.py:219-222) with one grouped kernel launch."""
    accumulate_modules(sow_modules(model), sync_reinit=sync_reinit)


def load_sow(model: nn.Module, checkpoint_path: str) -> None:
    """Load a safetensors checkpoint into a SoW model, growing empty accumulation parameters to their stored
    shape (prepare.py:188-215)."""
    from safetensors.torch import load_file
    tensors = load_file(checkpoint_path)
    own = model.state_dict()
    modules = dict(model.named_modules())
    for name, value in tensors.items():
        if name not in own:
            continue
        obj = model
        for part in name.split("."):
            obj = getattr(obj, part)
        if obj.numel() == 0:
            new = nn.Parameter(value.clone().to(_device_of(model)), requires_grad=False)
            if "." in name:
                parent, child = name.rsplit(".", 1)
                setattr(modules[parent], child, new)
            else:
                setattr(model, name, new)
        else:
            with torch.no_grad():
                obj.copy_(value.to(obj.device))        # in-place through the Parameter: bumps its version counter
    for m in sow_modules(model):                       # compute copies of W derived from the old values are stale now
        m._w_shadow = None
        m._w_shadow_key = None
    from .custom_ops import invalidate_weight_cache
    invalidate_weight_cache()


def _device_of(model: nn.Module) -> torch.device:
    for p in model.parameters():
        if p.numel():
            return p.device
    return torch.device("cpu")


def export_alignment(module, export_name, out_dir: Optional[str] = None):
    """Singular-vector alignment diagnostic (prepare.py:224-245).  The reference writes to a hard-coded home
    directory; here the directory is ``out_dir`` or $SOW_ALIGN_DIR or the current directory."""
    import numpy as np
    from .utils import svd_weight
    if not isinstance(module, SoWLinear):
        raise TypeError("Not a SoW layer")
    acc = None
    for a, b in zip(module.downscale_weights, module.upscale_weights):
        t = a.detach().float() @ b.detach().float()
        acc = t if acc is None else acc + t
    if module.acc_upweight.numel() != 0:
        weight = module.acc_downweight.float() @ module.acc_upweight.float()
    else:
        weight = module.acc_downweight.float()
    U_acc, _, _ = svd_weight(acc, module.rank)
    U_w, _, _ = svd_weight(weight)
    grid = torch.abs(U_w.T @ U_acc)
    pct = (grid / grid.sum(axis=0)) * 100
    out_dir = out_dir or os.environ.get("SOW_ALIGN_DIR", ".")
    path = os.path.join(out_dir, export_name + ".npy")
    np.save(path, pct.detach().cpu().numpy())
    return path
