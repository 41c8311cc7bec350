"""TEST INFRASTRUCTURE ONLY -- import the UNMODIFIED reference hot-path files from a checkout of the upstream project
(idonahum/photoVerse) named by the environment variable PHOTOVERSE_REFERENCE_ROOT.

The reference is pure Python; ``models/adapters.py`` needs only torch, ``models/attention_processor.py``
imports three diffusers symbols (attention_processor.py:5-9) that are absent from this image
(diffusers cannot be installed: no network).  We register a stub namespace for exactly those three
names and drive the verbatim file through a minimal stand-in for diffusers' ``Attention`` module
(fields listed in SURVEY.md §8b) and a stand-in for peft 0.10.0 ``lora.Linear``.

Nothing here is copied from the reference: the files are executed where they lie.  This module is
used only by ``oracle/make_golden.py`` and by the "live reference" legs of the tests; without a checkout the tests
compare against the reference outputs committed under ``tests/golden/``.
"""
import importlib.util
import os
import sys
import types

import torch
from torch import nn

REFERENCE_ROOT = os.environ.get("PHOTOVERSE_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "attention_processor.py"))


def _install_diffusers_stub():
    if "diffusers" in sys.modules and not getattr(sys.modules["diffusers"], "_pv_stub", False):
        return  # a real diffusers is importable; use it
    d = types.ModuleType("diffusers")
    d._pv_stub = True
    ip = types.ModuleType("diffusers.image_processor")
    ut = types.ModuleType("diffusers.utils")
    md = types.ModuleType("diffusers.models")
    ap = types.ModuleType("diffusers.models.attention_processor")

    class IPAdapterMaskProcessor:  # only referenced on the ip_adapter_masks path (never taken)
        @staticmethod
        def downsample(*a, **k):
            raise NotImplementedError("mask path is out of scope (SURVEY.md §2)")

    def deprecate(*a, **k):
        return None

    class Attention(nn.Module):  # annotation only in the reference signature
        pass

    ip.IPAdapterMaskProcessor = IPAdapterMaskProcessor
    ut.deprecate = deprecate
    ap.Attention = Attention
    d.image_processor, d.utils, d.models = ip, ut, md
    md.attention_processor = ap
    for name, mod in (("diffusers", d), ("diffusers.image_processor", ip), ("diffusers.utils", ut),
                      ("diffusers.models", md), ("diffusers.models.attention_processor", ap)):
        sys.modules[name] = mod


def _load(name: str, relpath: str):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_cache = {}


def load_reference_processor_module():
    if "proc" not in _cache:
        _install_diffusers_stub()
        _cache["proc"] = _load("_pv_ref_attention_processor", "models/attention_processor.py")
    return _cache["proc"]


def load_reference_adapter_module():
    if "adap" not in _cache:
        _cache["adap"] = _load("_pv_ref_adapters", "models/adapters.py")
    return _cache["adap"]


class LoraLinearStandIn(nn.Module):
    """peft 0.10.0 ``lora.Linear`` attribute layout + forward (restated, dependency not vendored):
    result = base_layer(x) + lora_B(lora_A(lora_dropout(x))) * scaling."""

    def __init__(self, base: nn.Linear, r: int, lora_alpha: float = 1.0, lora_dropout: float = 0.0):
        super().__init__()
        self.base_layer = base
        self.lora_A = nn.ModuleDict({"default": nn.Linear(base.in_features, r, bias=False)})
        self.lora_B = nn.ModuleDict({"default": nn.Linear(r, base.out_features, bias=False)})
        self.lora_dropout = nn.ModuleDict(
            {"default": nn.Dropout(lora_dropout) if lora_dropout > 0 else nn.Identity()})
        self.scaling = {"default": lora_alpha / r}
        self.r = {"default": r}

    @property
    def weight(self):
        return self.base_layer.weight

    def forward(self, x):
        y = self.base_layer(x)
        a, b = self.lora_A["default"], self.lora_B["default"]
        return y + b(a(self.lora_dropout["default"](x))) * self.scaling["default"]


class AttentionStandIn(nn.Module):
    """The subset of diffusers 0.27.2 ``Attention`` the reference processor touches for SD-1.5 attn2
    (attention_processor.py:275-305, :423-433)."""

    def __init__(self, query_dim: int, cross_attention_dim: int = 768, heads: int = 8):
        super().__init__()
        self.heads = heads
        self.to_q = nn.Linear(query_dim, query_dim, bias=False)
        self.to_k = nn.Linear(cross_attention_dim, query_dim, bias=False)
        self.to_v = nn.Linear(cross_attention_dim, query_dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(query_dim, query_dim, bias=True), nn.Dropout(0.0)])
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = None
        self.norm_encoder_hidden_states = None
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.scale = (query_dim // heads) ** -0.5
        self.processor = None

    def prepare_attention_mask(self, *a, **k):
        raise NotImplementedError("attention_mask is never passed on the PhotoVerse path")

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        return self.processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                              attention_mask=attention_mask, **kw)


def build_reference_layer(weights, dtype=torch.float32):
    """Instantiate the verbatim reference processor + Attention stand-in holding ``weights``
    (an oracle.processor_oracle.ProcessorWeights)."""
    mod = load_reference_processor_module()
    C = weights.to_q.shape[0]
    Dc = weights.to_k.shape[1]
    attn = AttentionStandIn(C, Dc, weights.heads)
    proc = mod.PhotoVerseAttnProcessor2_0(hidden_size=C, cross_attention_dim=Dc, num_tokens=(5,))
    attn.to(dtype)
    proc.to(dtype)
    with torch.no_grad():
        attn.to_q.weight.copy_(weights.to_q)
        attn.to_k.weight.copy_(weights.to_k)
        attn.to_v.weight.copy_(weights.to_v)
        attn.to_out[0].weight.copy_(weights.to_out_w)
        attn.to_out[0].bias.copy_(weights.to_out_b)
        proc.to_k_ip[0].weight.copy_(weights.to_k_ip)
        proc.to_v_ip[0].weight.copy_(weights.to_v_ip)
    for name, lw in weights.lora.items():
        base = getattr(attn, name)
        wrapped = LoraLinearStandIn(base, lw.A.shape[0], lora_alpha=lw.scaling * lw.A.shape[0]).to(dtype)
        with torch.no_grad():
            wrapped.lora_A["default"].weight.copy_(lw.A)
            wrapped.lora_B["default"].weight.copy_(lw.B)
        setattr(attn, name, wrapped)
    attn.processor = proc
    attn.to(dtype)
    return attn, proc


def load_reference_inject_fn():
    """The verbatim ``_inject_concept_embeddings`` of ``models/clip.py`` (:17-24).  The module itself does not import on
    the installed transformers (it needs 4.40 internals), so only that function's source is compiled, where it lies."""
    import ast
    path = os.path.join(REFERENCE_ROOT, "models", "clip.py")
    with open(path) as f:
        tree = ast.parse(f.read(), filename=path)
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "_inject_concept_embeddings")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    return ns["_inject_concept_embeddings"]


def load_reference_checkpoint_fns():
    """The verbatim ``save_progress`` and ``load_photoverse_model`` of ``models/modeling_utils.py`` (:13-50).  The module
    imports diffusers / peft / models.clip at the top (absent here), so only the two functions' sources are compiled,
    where they lie, against stand-ins for the two peft names they use:
      * ``LoraConfig``: a dataclass whose ``to_dict()`` is ``dataclasses.asdict`` like peft 0.10.0's PeftConfigMixin --
        including a ``peft_type`` enum member defined under peft's module path and ``target_modules`` as a set;
      * ``inject_adapter_in_model``: wraps the target Linears in LoraLinearStandIn.
    Returns (save_progress, load_photoverse_model, LoraConfig)."""
    import ast
    import dataclasses
    import enum
    path = os.path.join(REFERENCE_ROOT, "models", "modeling_utils.py")
    with open(path) as f:
        tree = ast.parse(f.read(), filename=path)
    fns = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ("save_progress", "load_photoverse_model")]
    assert len(fns) == 2

    # peft.utils.peft_types.PeftType, value == name (peft 0.10.0), pickled by reference under that module path
    mod = sys.modules.get("peft.utils.peft_types")
    if mod is None or not hasattr(mod, "PeftType"):
        peft = sys.modules.setdefault("peft", types.ModuleType("peft"))
        utils = sys.modules.setdefault("peft.utils", types.ModuleType("peft.utils"))
        mod = types.ModuleType("peft.utils.peft_types")
        mod.PeftType = enum.Enum("PeftType", {"LORA": "LORA", "IA3": "IA3"}, type=str, module="peft.utils.peft_types",
                                 qualname="PeftType")
        sys.modules["peft.utils.peft_types"] = mod
        peft.utils, utils.peft_types = utils, mod
    PeftType = mod.PeftType

    @dataclasses.dataclass
    class LoraConfig:
        r: int = 8
        lora_alpha: float = 8
        lora_dropout: float = 0.0
        target_modules: object = None
        init_lora_weights: bool = True
        peft_type: object = None
        task_type: object = None
        inference_mode: bool = False
        bias: str = "none"

        def __post_init__(self):
            self.peft_type = PeftType.LORA
            if isinstance(self.target_modules, list):
                self.target_modules = set(self.target_modules)

        def to_dict(self):
            return dataclasses.asdict(self)

    def inject_adapter_in_model(cfg, model):
        targets = tuple(cfg.target_modules)
        for name, module in list(model.named_modules()):
            for child_name, child in list(module.named_children()):
                qual = f"{name}.{child_name}" if name else child_name
                if isinstance(child, nn.Linear) and qual.endswith(targets):
                    setattr(module, child_name, LoraLinearStandIn(child, cfg.r, cfg.lora_alpha, cfg.lora_dropout))
        return model

    ns = {"torch": torch, "os": os, "LoraConfig": LoraConfig, "inject_adapter_in_model": inject_adapter_in_model}
    exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
    return ns["save_progress"], ns["load_photoverse_model"], LoraConfig
