"""TEST INFRASTRUCTURE ONLY -- the reference's out projection (attention_processor.py:423) with a peft 0.10.0
``lora.Linear`` on ``to_out[0]``, built on the oracle (oracle/processor_oracle.py), whose out projection is the plain
Linear of the reference's recipe.

:func:`dual_branch_attention_out_lora` evaluates the oracle with an identity out projection, which gives O, the input of
``to_out[0]``, and applies the oracle's ``lora_linear`` to it:  Y = O Wo^T + bo + s B_o A_o dropout(O).  The factors come
from ``w.lora["to_out"]`` and the keep-mask from ``drop["to_out"]``; without them it is the oracle itself.  Everything is
plain differentiable torch, so autograd through it is the checker of the backward too.
"""
import torch

from oracle.host_reference import OracleAttnProcessor, _parts, clone_with_oracle_processors
from oracle.processor_oracle import ProcessorWeights, dual_branch_attention, fusion_weights, lora_linear


def dual_branch_attention_out_lora(x, text, img, w: ProcessorWeights, w_text=1.0, w_img=1.0, drop=None):
    """Returns (Y [B,S,C], to_v_ip_norm [B,H,Li,1]) like ``dual_branch_attention``, with ``to_out`` LoRA-wrapped when
    ``w.lora`` has a ``"to_out"`` entry (its keep-mask, if any, drawn after those of to_q, to_k, to_v)."""
    drop = drop or {}
    lo = w.lora.get("to_out")
    if lo is None:
        return dual_branch_attention(x, text, img, w, w_text, w_img, drop)
    C = w.to_out_w.shape[0]
    eye = torch.eye(C, dtype=w.to_out_w.dtype, device=w.to_out_w.device)
    inner = ProcessorWeights(w.to_q, w.to_k, w.to_v, eye, torch.zeros_like(w.to_out_b), w.to_k_ip, w.to_v_ip, w.heads,
                             {k: v for k, v in w.lora.items() if k != "to_out"})
    o, vn = dual_branch_attention(x, text, img, inner, w_text, w_img, {k: v for k, v in drop.items() if k != "to_out"})
    return lora_linear(o, w.to_out_w, lo, drop.get("to_out")) + w.to_out_b, vn      # :423


class OutLoraOracleAttnProcessor(OracleAttnProcessor):
    """:class:`OracleAttnProcessor` that also reads a LoRA wrapper on ``attn.to_out[0]`` (eval-mode LoRA, no dropout)."""

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=2.0,
                 ip_adapter_masks=None):
        text, img = encoder_hidden_states
        if isinstance(img, list):
            img = img[0]
        cd = self.compute_dtype or hidden_states.dtype
        lora = {}
        parts = {}
        for name, mod in (("to_q", attn.to_q), ("to_k", attn.to_k), ("to_v", attn.to_v), ("to_out", attn.to_out[0])):
            parts[name], lw = _parts(mod)
            if lw:
                lora[name] = lw
        w = ProcessorWeights(parts["to_q"], parts["to_k"], parts["to_v"], parts["to_out"], attn.to_out[0].bias,
                             self.to_k_ip[0].weight, self.to_v_ip[0].weight, attn.heads, lora).to(dtype=cd)
        grad = torch.is_grad_enabled()
        u = torch.rand(1).item() if grad else None
        wt, wi = fusion_weights(grad, u, self.scale[0], self.fusion_rule1, self.fusion_rule2)
        y, vn = dual_branch_attention_out_lora(hidden_states.to(cd), text.to(cd), img.to(cd), w, wt, wi)
        self.to_v_ip_norm = vn.to(hidden_states.dtype)
        return y.to(hidden_states.dtype)


def clone_with_out_lora_oracle_processors(unet, device=None, dtype=None, compute_dtype=None):
    """:func:`clone_with_oracle_processors` whose oracle processors also apply a LoRA on ``to_out[0]``."""
    ref = clone_with_oracle_processors(unet, device, dtype, compute_dtype)
    for m in ref.modules():
        proc = getattr(m, "processor", None)
        if isinstance(proc, OracleAttnProcessor) and not isinstance(proc, OutLoraOracleAttnProcessor):
            op = OutLoraOracleAttnProcessor(proc.to_k_ip[0].weight.shape[0], proc.to_k_ip[0].weight.shape[1])
            op.to_k_ip[0].weight = proc.to_k_ip[0].weight
            op.to_v_ip[0].weight = proc.to_v_ip[0].weight
            op.compute_dtype = proc.compute_dtype
            m.set_processor(op)
    return ref

