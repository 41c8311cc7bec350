"""B200-native drop-in for the reference's ``models/attention_processor.py``.

``PhotoVerseAttnProcessor2_0`` keeps the reference's constructor, ``__call__`` signature, parameter names
(``to_k_ip.0.weight`` / ``to_v_ip.0.weight``), ``to_v_ip_norm`` side output and RNG consumption
(attention_processor.py:27-56, 236-254, 397, 411-420), so ``models/unet.py:set_visual_cross_attention_adapter``
and diffusers' ``Attention.forward`` can install and call it unchanged.  All arithmetic runs in the CUDA library
(photoverse_b200/csrc) through the C ABI; there is no PyTorch fallback.

Differences in *how* (not what) it computes, see DESIGN.md:
  * the two SDPA calls + add (:317-319, :400-402, :412) are one kernel: QK^T over the concatenated text+image keys,
    softmax normalised per segment, branch weights folded into P, one PV contraction;
  * LoRA on to_q/to_k/to_v and to_out[0] is merged into the packed bf16/fp16/fp32 weights on the GPU whenever a factor
    changes;
  * float16 models run the bf16 tensor-core kernels with fp16 operands (inference only: grad mode raises);
  * under CUDA autocast, float32 hidden states compute in the autocast dtype like the reference's autocast'd Linears and
    SDPA (bf16 always, fp16 without grad; DESIGN.md 4.9): float32 activations are converted by a native kernel;
  * K/V projections can be cached across denoising steps (``kv_cache`` context) because
    ``encoder_hidden_states`` is constant during generation (models/infer.py:89-98).
"""
import copy
from typing import Optional

import torch
from torch import nn

from . import ops
from .lora import linear_parts

_SUPPORTED = (torch.bfloat16, torch.float16, torch.float32)
_F16_TRAINING = ("float16 runs the inference (no_grad) path only: training runs in bfloat16 or float32 "
                 "(cast the model, or run the forward under torch.no_grad() without LoRA dropout)")


class PhotoVerseAttnProcessor(nn.Module):
    """Parameter container + constructor validation shared with the 2_0 class
    (reference attention_processor.py:27-56).  The legacy eager ``__call__`` of the reference
    (:58-218) is dead code on torch >= 2.0 (models/unet.py:26-28) and is not provided."""

    def __init__(self, hidden_size, cross_attention_dim=None, num_tokens=(5,), scale=2.0, fusion_rules=(1 / 3, 2 / 3)):
        super().__init__()
        self.hidden_size = hidden_size
        self.cross_attention_dim = cross_attention_dim
        if not isinstance(num_tokens, (tuple, list)):
            num_tokens = [num_tokens]
        self.num_tokens = num_tokens
        if not isinstance(fusion_rules, tuple) or len(fusion_rules) != 2 or not all(
                isinstance(i, float) for i in fusion_rules):
            raise ValueError("`fusion_rules` should be a tuple of two floats.")
        self.fusion_rule1, self.fusion_rule2 = fusion_rules
        if self.fusion_rule1 + self.fusion_rule2 != 1:
            raise ValueError("Sum of the fusion rules should be equal to 1.")
        if not isinstance(scale, list):
            scale = [scale] * len(num_tokens)
        if len(scale) != len(num_tokens):
            raise ValueError("`scale` should be a list of integers with the same length as `num_tokens`.")
        self.scale = scale
        self.to_k_ip = nn.ModuleList(
            [nn.Linear(cross_attention_dim, hidden_size, bias=False) for _ in range(len(num_tokens))])
        self.to_v_ip = nn.ModuleList(
            [nn.Linear(cross_attention_dim, hidden_size, bias=False) for _ in range(len(num_tokens))])

    def __call__(self, *args, **kwargs):
        raise NotImplementedError(
            "the pre-torch-2.0 eager processor is not part of the B200 path; use PhotoVerseAttnProcessor2_0")


class _PackedWeights:
    """Packed weights of one layer in one compute dtype.  Merged: LoRA folded into ``wq`` / ``wkv_text`` / ``wo``
    (W + s B A).  Unmerged (the LoRA-dropout training path): ``wq`` / ``wkv_text`` / ``wo`` hold the base weights and the
    low-rank branch is a K-extension of the base GEMM, ``[x | dropout(x) A^T] @ [W | s B]^T`` (``*_aug``, rank columns
    padded to 8)."""
    __slots__ = ("key", "wq", "wkv_text", "wkv_img", "wo", "bo", "_t",
                 "wq_aug", "wkv_text_aug", "wkv_img_aug", "wo_aug", "ranks", "eye")


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


class PhotoVerseAttnProcessor2_0(PhotoVerseAttnProcessor):
    def __init__(self, hidden_size, cross_attention_dim=None, num_tokens=(5,), scale=2.0, fusion_rules=(1 / 3, 2 / 3)):
        super().__init__(hidden_size, cross_attention_dim, num_tokens, scale, fusion_rules)
        self.to_v_ip_norm = None
        self._packed = {}          # (dtype, merged) -> _PackedWeights
        self._kv_cache = None      # dict while a kv_cache scope is active, else None
        self._kv_static = False
        self.last_fusion = (1.0, 1.0)

    # ------------------------------------------------------------------------------------------
    # K/V cache control (used by the denoise loop; off by default == reference behaviour)
    # ------------------------------------------------------------------------------------------
    def enable_kv_cache(self, enabled: bool = True, static: bool = False):
        """``static=True``: entries are keyed by buffer address only and live in persistent device buffers that
        :meth:`prepare_kv` refreshes in place -- what a captured CUDA graph needs (stable K/V addresses)."""
        self._kv_cache = {} if enabled else None
        self._kv_static = bool(static) and enabled

    def _kv_key(self, text, img, dtype):
        """Key of the caller's context tensors (not of their converted copies, which are new every call) and the compute
        dtype."""
        key = (text.data_ptr(), img.data_ptr(), tuple(text.shape), tuple(img.shape), text.dtype, img.dtype, dtype)
        if not getattr(self, "_kv_static", False):
            key += (text._version, img._version)
        return key

    @torch.no_grad()
    def prepare_kv(self, attn, text, img):
        """(Re)compute the packed K/V of this layer for the given contexts into the cache (in place when the
        entry exists).  Called once per generation by the denoise loop (SURVEY.md §0.1 D7).  The compute dtype is resolved
        from the text states like the processor resolves it from the hidden states (float32 under autocast: 16-bit)."""
        if self._kv_cache is None:
            raise RuntimeError("enable_kv_cache() first")
        autocast = ops.autocast_dtype() is not None
        dtype = ops.compute_dtype(text.dtype, False)
        pk = self._weights(attn, dtype, text.device)
        ck = self._kv_key(text, img, dtype)
        kv = ops.kv_pack(_cast(text, dtype, autocast, False), _cast(img, dtype, autocast, False), pk.wkv_text, pk.wkv_img,
                         attn.heads, out=self._kv_cache.get(ck))
        kv._keepalive = (text, img)
        self._kv_cache[ck] = kv
        return kv

    # ------------------------------------------------------------------------------------------
    def _weights(self, attn, dtype, device, merged: bool = True):
        """Packed weights of this layer in the compute dtype: LoRA merged (W + s B A), or with ``merged=False`` the base
        weights plus the K-extended operands of the LoRA-dropout path.  Each of the four operands is re-packed only when
        one of ITS OWN sources changed (parameter version counters): in training the optimizer touches the LoRA factors
        and to_k_ip / to_v_ip every step, the out projection only when it carries LoRA."""
        wq, qa, qb, qs, qp = linear_parts(attn.to_q)
        wk, ka, kb, ks, kp = linear_parts(attn.to_k)
        wv, va, vb, vs, vp = linear_parts(attn.to_v)
        wo, oa, ob, os_, op = linear_parts(attn.to_out[0])
        if merged and max(qp, kp, vp, op) > 0.0:
            raise RuntimeError("internal: merged weights requested while LoRA dropout is active")
        bo = attn.to_out[0].bias
        kip, vip = self.to_k_ip[0].weight, self.to_v_ip[0].weight

        def vkey(tensors, *scal):
            return tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors) + scal

        keys = {"wq": vkey([wq, qa, qb], qs), "wkv_text": vkey([wk, ka, kb, wv, va, vb], ks, vs),
                "wkv_img": vkey([kip, vip]), "wo": vkey([wo, bo, oa, ob], os_)}
        pk = self._packed.get((dtype, merged))
        if pk is not None and pk.key == keys:
            return pk
        C, Dc = wq.shape[0], wk.shape[1]
        for t in (wq, qa, qb, wk, ka, kb, wv, va, vb, wo, oa, ob, bo, kip, vip):
            if t is not None and not t.is_cuda:
                raise RuntimeError(f"photoverse_b200 needs its weights on the CUDA device (got {t.device})")

        def m(t):   # fp32 master view of a parameter (a cast happens only if the module was .to(bf16)'d)
            return None if t is None else t.detach().float().contiguous()

        def lora(a, b, s):     # the LoRA operands of pack_weight: none when the branch stays a K-extension
            return (m(a), m(b), s) if merged else ()

        def sb(b, s, r8):      # s * B, rank columns zero-padded to r8 (weight layout only, no activation math)
            out = torch.zeros(C, r8, device=device, dtype=dtype)
            out[:, :b.shape[1]] = (b.detach().float() * s).to(dtype)
            return out

        old = pk.key if pk is not None else {}
        fresh = {name for name in keys if old.get(name) != keys[name]}
        with torch.no_grad():
            if pk is None:
                pk = _PackedWeights()
                pk._t = {}
                # bf16: the attention kernel always applies a [C,C] projection; the already-projected Q goes through I
                pk.eye = torch.eye(C, device=device, dtype=dtype) if dtype == torch.bfloat16 and not merged else None
            else:                      # a NEW object per key set: autograd contexts of earlier calls keep the old one
                pk = copy.copy(pk)
                pk._t = dict(pk._t)
            if "wq" in fresh:
                pk.wq = ops.pack_weight(m(wq), torch.empty(C, C, device=device, dtype=dtype), *lora(qa, qb, qs))
                pk._t.pop("wq_t", None)
            if "wkv_text" in fresh:
                pk.wkv_text = torch.empty(2 * C, Dc, device=device, dtype=dtype)
                ops.pack_weight(m(wk), pk.wkv_text[:C], *lora(ka, kb, ks))
                ops.pack_weight(m(wv), pk.wkv_text[C:], *lora(va, vb, vs))
                pk._t.pop("wkv_text_t", None)
            if "wkv_img" in fresh:
                pk.wkv_img = torch.empty(2 * C, Dc, device=device, dtype=dtype)
                ops.pack_weight(m(kip), pk.wkv_img[:C])
                ops.pack_weight(m(vip), pk.wkv_img[C:])
                pk._t.pop("wkv_img_t", None)
            if "wo" in fresh:
                pk.wo = ops.pack_weight(m(wo), torch.empty(C, C, device=device, dtype=dtype), *lora(oa, ob, os_))
                pk.bo = m(bo) if bo is not None else torch.zeros(C, device=device, dtype=torch.float32)
                pk._t.pop("wo_t", None)
            if not merged:
                pk.ranks = rq, rk, rv, ro = tuple(0 if a is None else _pad8(a.shape[0]) for a in (qa, ka, va, oa))
                if "wq" in fresh:
                    pk.wq_aug = torch.cat([pk.wq, sb(qb, qs, rq)], 1).contiguous() if rq else pk.wq
                if "wo" in fresh:
                    pk.wo_aug = torch.cat([pk.wo, sb(ob, os_, ro)], 1).contiguous() if ro else pk.wo
                if fresh & {"wkv_text", "wkv_img"}:
                    if rk or rv:       # K/V of the text branch with their low-rank columns, image branch zero-extended
                        ext = torch.zeros(2 * C, rk + rv, device=device, dtype=dtype)
                        if rk:
                            ext[:C, :rk] = sb(kb, ks, rk)
                        if rv:
                            ext[C:, rk:] = sb(vb, vs, rv)
                        pk.wkv_text_aug = torch.cat([pk.wkv_text, ext], 1).contiguous()
                        pk.wkv_img_aug = torch.cat([pk.wkv_img, torch.zeros_like(ext)], 1).contiguous()
                    else:
                        pk.wkv_text_aug, pk.wkv_img_aug = pk.wkv_text, pk.wkv_img
            pk.key = keys
        self._packed[(dtype, merged)] = pk
        if self._kv_cache is not None and fresh & {"wkv_text", "wkv_img"}:
            self._kv_cache.clear()
        return pk

    def lora_dropout_active(self, attn) -> bool:
        """True when a LoRA-wrapped projection of ``attn`` is in training mode with dropout p > 0 (peft applies
        ``lora_dropout`` to the low-rank branch input only; train.py:264-269, 348-354)."""
        return any(linear_parts(m)[4] > 0.0 for m in (attn.to_q, attn.to_k, attn.to_v, attn.to_out[0]))

    def _fusion_weights(self):
        """(w_text, w_image) -- reference attention_processor.py:411-420, including its RNG draw."""
        if not torch.is_grad_enabled():
            return 1.0, 1.0
        seed = torch.rand(1).item()          # exactly one draw from the global CPU generator per call
        scale = self.scale[0]
        if isinstance(scale, (list, tuple)):
            scale = scale[0]
        if seed < self.fusion_rule1:
            return float(scale), 0.0
        if seed > self.fusion_rule2:
            return 0.0, float(scale)
        return 1.0, 1.0

    def __call__(
        self,
        attn,
        hidden_states: torch.Tensor,
        encoder_hidden_states=None,
        attention_mask: Optional[torch.Tensor] = None,
        temb: Optional[torch.Tensor] = None,
        scale: float = 2.0,
        ip_adapter_masks=None,
    ):
        # ---- unpack (reference :258-273) ----
        if encoder_hidden_states is None:
            raise ValueError("PhotoVerseAttnProcessor2_0 is a cross-attention processor: encoder_hidden_states "
                             "must be (text, image) ")
        if isinstance(encoder_hidden_states, tuple):
            encoder_hidden_states, ip_hidden_states = encoder_hidden_states
            if not isinstance(ip_hidden_states, list):
                ip_hidden_states = [ip_hidden_states]
        else:  # deprecated tensor form: the last num_tokens[0] rows are the image tokens
            end_pos = encoder_hidden_states.shape[1] - self.num_tokens[0]
            encoder_hidden_states, ip_hidden_states = (
                encoder_hidden_states[:, :end_pos, :], [encoder_hidden_states[:, end_pos:, :]])
        if len(ip_hidden_states) != 1 or len(self.to_k_ip) != 1:
            raise NotImplementedError("PhotoVerse installs exactly one image adapter per layer (models/unet.py:29-33)")
        # ---- features of diffusers' Attention that are inactive for SD-1.5 attn2: refuse, never fall back ----
        if attention_mask is not None or ip_adapter_masks is not None:
            raise NotImplementedError("attention_mask / ip_adapter_masks are never passed on the PhotoVerse path")
        if hidden_states.ndim != 3:
            raise NotImplementedError("only [B, S, C] hidden states (SD-1.5 attn2) are supported")
        if getattr(attn, "spatial_norm", None) is not None or getattr(attn, "group_norm", None) is not None \
                or getattr(attn, "norm_cross", None):
            raise NotImplementedError("spatial_norm / group_norm / norm_cross are not part of the SD-1.5 attn2 path")
        if getattr(attn, "residual_connection", False) or getattr(attn, "rescale_output_factor", 1.0) != 1.0:
            raise NotImplementedError("residual_connection / rescale_output_factor != 1 unsupported")
        if hidden_states.dtype not in _SUPPORTED:
            raise TypeError(f"hidden_states must be bfloat16, float16 or float32, got {hidden_states.dtype}")
        if not hidden_states.is_cuda:
            raise RuntimeError("photoverse_b200 runs on CUDA only (no CPU fallback)")

        dev = hidden_states.device
        text_in, img_in = encoder_hidden_states, ip_hidden_states[0]
        w_text, w_img = self._fusion_weights()
        self.last_fusion = (w_text, w_img)

        train = (torch.is_grad_enabled() and (
            hidden_states.requires_grad or text_in.requires_grad or img_in.requires_grad
            or any(p.requires_grad for p in self.parameters())
            or any(p.requires_grad for m in (attn.to_q, attn.to_k, attn.to_v, attn.to_out[0]) for p in m.parameters()))
        ) or self.lora_dropout_active(attn)
        # the hidden states decide the compute dtype (DESIGN.md 4.9); under CUDA autocast a float32 X computes in 16 bits
        autocast = ops.autocast_dtype() is not None
        dtype = ops.compute_dtype(hidden_states.dtype, train)
        if train:
            if dtype == torch.float16:
                raise NotImplementedError(_F16_TRAINING)
            from .autograd import dual_attn_autograd
            x, text, img = (_cast(t, dtype, autocast, True) for t in (hidden_states, text_in, img_in))
            y, vnorm = dual_attn_autograd(self, attn, x, text, img, w_text, w_img)
            # side output (:397): [B, H, Li, 1] in the activation dtype, float32 under autocast (torch.norm's autocast dtype)
            self.to_v_ip_norm = (vnorm if autocast else vnorm.to(dtype)).unsqueeze(-1)
            return y

        x = _cast(hidden_states, dtype, autocast, False)
        pk = self._weights(attn, dtype, dev)
        kv = None
        ck = None
        if self._kv_cache is not None:
            ck = self._kv_key(text_in, img_in, dtype)
            kv = self._kv_cache.get(ck)
        if kv is None:
            text, img = _cast(text_in, dtype, autocast, False), _cast(img_in, dtype, autocast, False)
            kv = ops.kv_pack(text, img, pk.wkv_text, pk.wkv_img, attn.heads)
            if self._kv_cache is not None:
                kv._keepalive = (text_in, img_in)      # pin the storage so the data_ptr key cannot be recycled
                self._kv_cache[ck] = kv
        y, _, _, _ = ops.dual_attn(x, pk.wq, kv, pk.wo, pk.bo, w_text, w_img)
        # side output (:397): [B, H, Li, 1] in the activation dtype, float32 under autocast
        self.to_v_ip_norm = kv.v_ip_norm.unsqueeze(-1) if autocast else kv.vnorm_act
        return y


def _cast(t: torch.Tensor, dtype: torch.dtype, autocast: bool, grad: bool) -> torch.Tensor:
    """``t`` as a contiguous tensor of the compute dtype.  Under autocast a float32 <-> 16-bit conversion is the native
    kernel (differentiable in grad mode); outside autocast, and between the two 16-bit types, it stays ``Tensor.to``."""
    if t.dtype == dtype:
        return t.contiguous()
    if autocast and torch.float32 in (t.dtype, dtype):
        if grad:
            from .autograd import convert
            return convert(t, dtype)
        return ops.convert(t, dtype)
    return t.to(dtype).contiguous()
