"""LoRA on the cross-attention projections (reference: train.py:348-354, models/modeling_utils.py:86-88).

The reference injects peft==0.10.0 ``lora.Linear`` wrappers into ``attn2.to_q / to_k / to_v``; ``attn2.to_out.0`` (the
usual diffusers target set adds it) is supported as a fourth target in inference and training.  peft is not
installable here, so this module provides a wrapper with the SAME attribute layout and state-dict key names
(``base_layer.weight``, ``lora_A.default.weight``, ``lora_B.default.weight``, ``scaling['default']``,
``lora_dropout.default``) so that reference checkpoints (modeling_utils.py:29-50) load unchanged, and the
B200 processor reads the factors straight out of whichever wrapper (ours or real peft) it finds.

The wrapper never does arithmetic on the hot path: the processor merges W + scaling*B*A inside
``pv_pack_weight`` (CUDA) whenever a factor's version counter changes.  Only ``attn2`` modules can be targets: the host
UNet runs ``attn1`` and the feed-forward layers as stock modules, which would call :meth:`LoraLinear.forward` (it
raises), so write the targets with the ``attn2.`` prefix.
"""
import math
from typing import Iterable, Optional, Tuple

import torch
from torch import nn

DEFAULT_TARGETS = ("attn2.to_k", "attn2.to_v", "attn2.to_q")      # train.py:353


class LoraLinear(nn.Module):
    def __init__(self, base_layer: nn.Linear, r: int = 8, lora_alpha: float = 1.0, lora_dropout: float = 0.0):
        super().__init__()
        if r <= 0:
            raise ValueError("`r` should be a positive integer value")
        self.base_layer = base_layer
        self.in_features, self.out_features = base_layer.in_features, base_layer.out_features
        dev, dt = base_layer.weight.device, base_layer.weight.dtype
        self.lora_A = nn.ModuleDict({"default": nn.Linear(self.in_features, r, bias=False, device=dev, dtype=dt)})
        self.lora_B = nn.ModuleDict({"default": nn.Linear(r, self.out_features, bias=False, device=dev, dtype=dt)})
        self.lora_dropout = nn.ModuleDict(
            {"default": nn.Dropout(p=lora_dropout) if lora_dropout > 0.0 else nn.Identity()})
        self.scaling = {"default": lora_alpha / r}
        self.r = {"default": r}
        self.lora_alpha = {"default": lora_alpha}
        # peft init: A kaiming-uniform(a=sqrt(5)), B zeros -> a freshly injected LoRA is an exact no-op
        nn.init.kaiming_uniform_(self.lora_A["default"].weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B["default"].weight)
        base_layer.weight.requires_grad_(False)     # peft freezes everything that is not lora_*

    @property
    def weight(self) -> torch.Tensor:
        return self.base_layer.weight

    @property
    def bias(self):
        return self.base_layer.bias

    def forward(self, x):  # pragma: no cover - the B200 processor never calls the wrapper
        raise RuntimeError("photoverse_b200.LoraLinear is a parameter container; the CUDA processor merges the "
                           "low-rank update itself (no PyTorch fallback path)")


def linear_parts(mod) -> Tuple[torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor], float, float]:
    """(W, lora_A|None, lora_B|None, scaling, dropout_p) of a plain ``nn.Linear`` or a peft-style wrapper."""
    if hasattr(mod, "base_layer") and hasattr(mod, "lora_A"):
        name = "default"
        A = mod.lora_A[name].weight
        B = mod.lora_B[name].weight
        scaling = float(mod.scaling[name])
        drop = mod.lora_dropout[name] if name in mod.lora_dropout else None
        p = float(getattr(drop, "p", 0.0)) if (drop is not None and mod.training) else 0.0
        return mod.base_layer.weight, A, B, scaling, p
    return mod.weight, None, None, 0.0, 0.0


def inject_lora(unet: nn.Module, r: int = 8, lora_alpha: float = 1.0, lora_dropout: float = 0.0,
                target_modules: Iterable[str] = DEFAULT_TARGETS) -> nn.Module:
    """Counterpart of ``peft.inject_adapter_in_model(LoraConfig(...), unet)`` for the reference's config:
    wraps every module whose qualified name ends with one of ``target_modules`` and freezes all parameters whose
    name does not contain ``lora_`` (peft semantics; SURVEY.md §0.1 D8)."""
    targets = tuple(target_modules)
    for name, module in list(unet.named_modules()):
        for child_name, child in list(module.named_children()):
            qual = f"{name}.{child_name}" if name else child_name
            if isinstance(child, nn.Linear) and qual.endswith(targets):
                setattr(module, child_name, LoraLinear(child, r, lora_alpha, lora_dropout))
    for pname, p in unet.named_parameters():
        if "lora_" not in pname:
            p.requires_grad_(False)
    return unet
