"""PhotoVerse checkpoint wire format (counterpart of reference ``models/modeling_utils.py:13-50``; SURVEY 8 f3).

One ``torch.save`` dict:
    "image_adapter" / "text_adapter"   adapter state dicts (``mapping_{i}.{0,1,3,4,6}.{weight,bias}``)
    "cross_attention_adapter"          every unet key that contains "attn2" AND one of "processor", "to_q", "to_k",
                                       "to_v" -- i.e. ``...attn2.processor.to_k_ip.0.weight`` plus, with LoRA, the peft
                                       keys ``...attn2.to_q.base_layer.weight / lora_A.default.weight / lora_B.default.weight``;
                                       and the keys of ``attn2.to_out.0`` when it is LoRA-wrapped (``...attn2.to_out.0.
                                       base_layer.weight / base_layer.bias / lora_A.default.weight / lora_B.default.weight``)
    "optimizer" (optional), "lora_config" (optional dict: r, lora_alpha, lora_dropout, target_modules)
Files written by the reference load here (tests/test_host_logic.py::test_checkpoint_written_by_the_reference_loads:
a file produced by the verbatim ``save_progress`` with a peft-0.10-shaped ``lora_config`` -- enum + set included) and
files written here are plain-typed, so the reference's loader reads them (host-side dict handling only; no arithmetic).
"""
import enum
import os
from typing import Optional

import torch

from .lora import DEFAULT_TARGETS, LoraLinear, inject_lora


# ---- reading files the reference wrote ---------------------------------------------------------------------------
# The reference stores ``lora_config.to_dict()`` (modeling_utils.py:45-46), which for peft 0.10.0 is ``asdict()`` of the
# LoraConfig dataclass: it contains ``peft.utils.peft_types.PeftType`` / ``TaskType`` enum members and a ``set``
# (target_modules).  ``torch.load`` unpickles with ``weights_only=True`` by default and refuses those enum globals; peft
# itself need not be installed where the file is read.  The two enums are therefore described here (value == name, as in
# peft) under peft's own module path and handed to torch's allowlist for the duration of the load -- nothing else is
# unpickled outside torch's weights-only rules.
def _peft_enum(name: str, members):
    cls = enum.Enum(name, {m: m for m in members}, type=str, module="peft.utils.peft_types", qualname=name)
    return cls


_PeftType = _peft_enum("PeftType", ("PROMPT_TUNING", "MULTITASK_PROMPT_TUNING", "P_TUNING", "PREFIX_TUNING", "LORA", "ADALORA",
                                    "BOFT", "ADAPTION_PROMPT", "IA3", "LOHA", "LOKR", "OFT", "POLY", "LN_TUNING", "VERA"))
_TaskType = _peft_enum("TaskType", ("SEQ_CLS", "SEQ_2_SEQ_LM", "CAUSAL_LM", "TOKEN_CLS", "QUESTION_ANS", "FEATURE_EXTRACTION"))


def _plain(v):
    """Enum -> its value, set / tuple -> sorted list / list, recursively: a config of plain JSON-like types."""
    if isinstance(v, enum.Enum):
        return _plain(v.value)
    if isinstance(v, (set, frozenset)):
        return sorted(_plain(x) for x in v)
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    if isinstance(v, dict):
        return {k: _plain(x) for k, x in v.items()}
    return v


def normalise_lora_config(cfg) -> Optional[dict]:
    """A peft ``LoraConfig`` (``to_dict()``), the dict the reference stored, or a plain dict -> plain-typed dict."""
    if cfg is None:
        return None
    if hasattr(cfg, "to_dict"):
        cfg = cfg.to_dict()
    return _plain(dict(cfg))


def read_checkpoint(path: str) -> dict:
    """``torch.load`` of a PhotoVerse ``.pt`` (ours or the reference's) under weights-only rules + the two peft enums."""
    try:
        real = []
        try:                                     # a real peft install: allow its own classes as well
            from peft.utils.peft_types import PeftType, TaskType  # type: ignore
            real = [PeftType, TaskType]
        except Exception:
            pass
        with torch.serialization.safe_globals([_PeftType, _TaskType] + real):
            return torch.load(path, map_location="cpu", weights_only=True)
    except Exception as e:  # noqa: BLE001 -- report what the file contains instead of a bare unpickling error
        raise RuntimeError(
            f"{path}: not readable as a PhotoVerse checkpoint under torch.load(weights_only=True) "
            f"(+ peft PeftType/TaskType): {e}") from e


def cross_attention_state_dict(unet) -> dict:
    """The reference's attn2 key filter (modeling_utils.py:29-50), plus a LoRA-wrapped ``attn2.to_out.0``: the reference
    trains no out-projection LoRA, so its filter has no term for one, but a trained one must survive a save and load."""
    out_lora = tuple(f"{name}." for name, m in unet.named_modules()
                     if name.endswith("attn2.to_out.0") and hasattr(m, "base_layer") and hasattr(m, "lora_A"))
    out = {}
    for key, value in unet.state_dict().items():
        if ("attn2" in key and ("processor" in key or "to_q" in key or "to_k" in key or "to_v" in key)) \
                or key.startswith(out_lora):
            out[key] = value
    return out


def save_progress(image_adapter, text_adapter, unet, output_path: str, step: Optional[int] = None,
                  lora_config: Optional[dict] = None, optimizer=None) -> str:
    final = {"image_adapter": image_adapter.state_dict(), "text_adapter": text_adapter.state_dict(),
             "cross_attention_adapter": cross_attention_state_dict(unet)}
    if optimizer is not None:
        final["optimizer"] = optimizer.state_dict()
    if lora_config is not None:
        # plain types (enum -> str, set -> list): loads everywhere under weights_only=True, and peft's
        # ``LoraConfig(**cfg)`` in the reference's loader (modeling_utils.py:16-18) accepts it unchanged
        final["lora_config"] = normalise_lora_config(lora_config)
    name = f"photoverse_{str(step).zfill(6)}.pt" if step is not None else "photoverse.pt"
    path = os.path.join(output_path, name)
    torch.save(final, path)
    return path


def load_photoverse_model(path: str, image_adapter, text_adapter, unet):
    """Returns (image_adapter, text_adapter, unet, lora_config) like the reference; injects LoRA wrappers first when
    the checkpoint carries a ``lora_config`` and the unet has none yet."""
    sd = read_checkpoint(path)
    lora_config = normalise_lora_config(sd.get("lora_config"))
    if lora_config is not None and not any(isinstance(m, LoraLinear) for m in unet.modules()):
        targets = lora_config.get("target_modules") or DEFAULT_TARGETS
        if isinstance(targets, str):
            targets = [targets]
        inject_lora(unet, r=int(lora_config.get("r", 8)), lora_alpha=float(lora_config.get("lora_alpha", 1.0)),
                    lora_dropout=float(lora_config.get("lora_dropout", 0.0)), target_modules=tuple(targets))
    if "image_adapter" in sd:
        image_adapter.load_state_dict(sd["image_adapter"])
    if "text_adapter" in sd:
        text_adapter.load_state_dict(sd["text_adapter"])
    if "cross_attention_adapter" in sd:
        unet.load_state_dict(sd["cross_attention_adapter"], strict=False)
    return image_adapter, text_adapter, unet, lora_config
