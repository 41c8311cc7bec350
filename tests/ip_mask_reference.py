"""TEST INFRASTRUCTURE ONLY -- regional identity masks (diffusers' ``ip_adapter_masks``) on top of the oracle
(oracle/processor_oracle.py).

:func:`downsample` restates diffusers 0.27.2 ``IPAdapterMaskProcessor.downsample(mask, batch_size, num_queries,
value_embed_dim)`` (diffusers/image_processor.py) for one adapter, without the final repeat over the value dimension:

    o_h, o_w = mask.shape[1], mask.shape[2];  ratio = o_w / o_h
    mask_h = int(sqrt(num_queries / ratio));  mask_h += (num_queries % mask_h != 0);  mask_w = num_queries // mask_h
    F.interpolate(mask.unsqueeze(0), size=(mask_h, mask_w), mode="bicubic").squeeze(0)    (align_corners=False)
    repeat(batch_size, 1, 1) when the mask batch is smaller;  view(batch, -1);  F.pad(..., value=0) to num_queries or
    [:, :num_queries]

:func:`masked_attention` is the masked output of diffusers' IPAdapterAttnProcessor2_0 for one image branch:
``O = w_text softmax(Q K_t^T/sqrt d) V_t + w_img m[b, s] softmax(Q K_i^T/sqrt d) V_i``, ``Y = O Wo^T + bo`` (with the
LoRA on to_out of tests/lora_out_reference.py when ``w.lora`` has one).  The reference's masked branch
(attention_processor.py:324-390) is diffusers' code copied verbatim and no PhotoVerse caller reaches it, so the golden
vectors pinned against the reference do not cover it: this restatement is the checker.  With ``m`` = None it is the oracle
itself.  Everything is plain differentiable torch (the mask gets no gradient).
"""
import math

import torch
import torch.nn.functional as F

from oracle.host_reference import OracleAttnProcessor, _parts, clone_with_oracle_processors
from oracle.processor_oracle import ProcessorWeights, dual_branch_attention, fusion_weights, lora_linear


def grid(S: int, H_m: int, W_m: int):
    ratio = W_m / H_m
    mask_h = int(math.sqrt(S / ratio))
    mask_h = int(mask_h) + int((S % int(mask_h)) != 0)
    return mask_h, S // mask_h


def downsample(mask: torch.Tensor, batch_size: int, S: int) -> torch.Tensor:
    """mask [1|B, H_m, W_m] -> [batch_size, S] in float64."""
    mask = mask.double()
    mask_h, mask_w = grid(S, mask.shape[1], mask.shape[2])
    md = F.interpolate(mask.unsqueeze(0), size=(mask_h, mask_w), mode="bicubic").squeeze(0)
    if md.shape[0] < batch_size:
        md = md.repeat(batch_size, 1, 1)
    md = md.view(md.shape[0], -1)
    if mask_h * mask_w < S:
        md = F.pad(md, (0, S - md.shape[1]), value=0.0)
    if mask_h * mask_w > S:
        md = md[:, :S]
    return md


def masked_attention(x, text, img, w: ProcessorWeights, w_text=1.0, w_img=1.0, m=None, drop=None):
    """(Y [B,S,C], to_v_ip_norm [B,H,Li,1]); ``m`` [B, S] row weights of the image branch (None: unmasked)."""
    drop = drop or {}
    inner_drop = {k: v for k, v in drop.items() if k != "to_out"}
    C = w.to_out_w.shape[0]
    eye = torch.eye(C, dtype=w.to_out_w.dtype, device=w.to_out_w.device)
    inner = ProcessorWeights(w.to_q, w.to_k, w.to_v, eye, torch.zeros_like(w.to_out_b), w.to_k_ip, w.to_v_ip, w.heads,
                             {k: v for k, v in w.lora.items() if k != "to_out"})
    if m is None:
        o, vn = dual_branch_attention(x, text, img, inner, w_text, w_img, inner_drop)
    else:
        o_t, vn = dual_branch_attention(x, text, img, inner, w_text, 0.0, inner_drop)
        o_i, _ = dual_branch_attention(x, text, img, inner, 0.0, w_img, inner_drop)
        o = o_t + m.to(o_i.dtype).unsqueeze(-1) * o_i
    return lora_linear(o, w.to_out_w, w.lora.get("to_out"), drop.get("to_out")) + w.to_out_b, vn


class MaskedOracleAttnProcessor(OracleAttnProcessor):
    """:class:`OracleAttnProcessor` that applies ``ip_adapter_masks`` by :func:`downsample` / :func:`masked_attention`."""

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=2.0,
                 ip_adapter_masks=None):
        text, img = encoder_hidden_states
        if isinstance(img, list):
            img = img[0]
        cd = self.compute_dtype or hidden_states.dtype
        lora, parts = {}, {}
        for name, mod in (("to_q", attn.to_q), ("to_k", attn.to_k), ("to_v", attn.to_v), ("to_out", attn.to_out[0])):
            parts[name], lw = _parts(mod)
            if lw:
                lora[name] = lw
        w = ProcessorWeights(parts["to_q"], parts["to_k"], parts["to_v"], parts["to_out"], attn.to_out[0].bias,
                             self.to_k_ip[0].weight, self.to_v_ip[0].weight, attn.heads, lora).to(dtype=cd)
        grad = torch.is_grad_enabled()
        u = torch.rand(1).item() if grad else None
        wt, wi = fusion_weights(grad, u, self.scale[0], self.fusion_rule1, self.fusion_rule2)
        B, S, _ = hidden_states.shape
        m = None
        if ip_adapter_masks is not None:
            m = downsample(ip_adapter_masks[0][:, 0], B, S).to(device=hidden_states.device, dtype=cd)
        y, vn = masked_attention(hidden_states.to(cd), text.to(cd), img.to(cd), w, wt, wi, m)
        self.to_v_ip_norm = vn.to(hidden_states.dtype)
        return y.to(hidden_states.dtype)


def clone_with_masked_oracle_processors(unet, device=None, dtype=None, compute_dtype=None):
    ref = clone_with_oracle_processors(unet, device, dtype, compute_dtype)
    for mod in ref.modules():
        proc = getattr(mod, "processor", None)
        if isinstance(proc, OracleAttnProcessor):
            op = MaskedOracleAttnProcessor(proc.to_k_ip[0].weight.shape[0], proc.to_k_ip[0].weight.shape[1])
            op.to_k_ip[0].weight = proc.to_k_ip[0].weight
            op.to_v_ip[0].weight = proc.to_v_ip[0].weight
            op.compute_dtype = proc.compute_dtype
            mod.set_processor(op)
    return ref
