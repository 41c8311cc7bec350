"""Host model: a Stable-Diffusion-1.5-shaped UNet in plain PyTorch (random-init; diffusers is not installable here).

This is NOT part of the B200 hot path -- it is the *caller* of the path (SURVEY.md §8 f1): the backbone the
PhotoVerse processors are plugged into so that images/s can be measured.  ResNet blocks, self-attention (attn1),
GEGLU feed-forward, up/down-sampling run as stock PyTorch / cuDNN library code on both the reference arm and ours;
only the 16 ``attn2`` layers go through photoverse_b200's kernels.

It reproduces diffusers 0.27.2's ``UNet2DConditionModel`` for the SD-1.5 config (module tree, parameter names,
``attn_processors`` / ``set_attn_processor`` / ``config`` protocol, processor key names consumed by the reference's
``models/unet.py:10-19``) so the reference's installation code and checkpoints' key layout apply unchanged.
"""
import math
from types import SimpleNamespace
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F
from torch import nn


# Epilogues of the backbone as photoverse_b200 kernels (csrc/pv_backbone.cu): GroupNorm (+ SiLU) directly on the
# channels-last activation (the stock sequence is NHWC -> NCHW copy, moments, normalise, SiLU, NCHW -> NHWC copy), LayerNorm,
# the GEGLU product, bias / residual sums -- the glue that was half of a generation step's GPU time.  Used for CUDA bf16
# channels-last activations: plain calls with autograd off, torch.autograd.Functions with an input-gradient kernel with
# autograd on when the module's affine is frozen (the PhotoVerse training set never includes the backbone); fp32 parity
# runs, NCHW models and trainable norms keep the stock PyTorch ops.  ``FUSED_EPILOGUES = False`` restores the stock
# sequence everywhere; ``UNetSD15.set_fused_epilogues(False)`` does so for one model (bench.py --stock-epilogues; the
# oracle arm of the parity tests; tests compare the two).
FUSED_EPILOGUES = True


def _enabled(mod: nn.Module, x: torch.Tensor) -> bool:
    return FUSED_EPILOGUES and getattr(mod, "_pv_fused", True) and x.is_cuda and x.dtype == torch.bfloat16


def _fused(mod: nn.Module, x: torch.Tensor) -> bool:
    """The inference-only kernels (LayerNorm, GEGLU) apply."""
    return _enabled(mod, x) and not torch.is_grad_enabled()


def _frozen(*tensors) -> bool:
    return not any(t is not None and t.requires_grad for t in tensors)


def _f32_params(mod: nn.Module, *names):
    """fp32 copies of a module's (bf16) parameters for the kernels' affine terms, refreshed when a parameter changes."""
    ps = [getattr(mod, n) for n in names]
    key = tuple((p.data_ptr(), p._version) for p in ps)
    cached = getattr(mod, "_pv_f32", None)
    if cached is None or cached[0] != key:
        cached = (key, [p.detach().float().contiguous() for p in ps])
        mod._pv_f32 = cached
    return cached[1]


def _nhwc(x: torch.Tensor) -> bool:
    return (x.dim() == 4 and x.shape[1] % 8 == 0 and x.shape[1] <= 4096 and x.is_contiguous(memory_format=torch.channels_last)
            and not x.is_contiguous())


class _GroupNormActFn(torch.autograd.Function):
    """Training-time ``[silu](norm(x))`` on a channels-last activation with a FROZEN affine (the PhotoVerse training set is
    adapters + to_k_ip / to_v_ip + LoRA factors, train.py:348-370): forward and input gradient are two launches each
    (csrc/pv_backbone.cu) instead of the stock copy / moments / normalise / SiLU / copy chain and its backward; only x and
    the per-(sample, group) statistics are kept."""

    @staticmethod
    def forward(ctx, x, add, gamma, beta, groups, eps, silu):
        from .. import ops
        y, stats = ops.group_norm_nhwc(x, gamma, beta, groups, eps, silu, add, save_stats=True)
        ctx.save_for_backward(x, stats, gamma, beta, *([] if add is None else [add]))
        ctx.cfg = (groups, silu)
        return y

    @staticmethod
    def backward(ctx, dy):
        from .. import ops
        x, stats, gamma, beta, *rest = ctx.saved_tensors
        dy = dy.contiguous(memory_format=torch.channels_last)
        dx = ops.group_norm_nhwc_bwd(x, dy, stats, gamma, beta, *ctx.cfg, add=rest[0] if rest else None)
        return dx, None, None, None, None, None, None        # the addend (conv bias + temb of a frozen backbone) has no gradient


class _AddBiasFn(torch.autograd.Function):
    """``a + b + bias[c]`` (frozen bias) in one pass; the gradient of both operands is the incoming gradient."""

    @staticmethod
    def forward(ctx, a, b, bias):
        from .. import ops
        return ops.add_bias_nhwc(a, b, bias)

    @staticmethod
    def backward(ctx, dy):
        return dy, dy, None


def group_norm_act(norm: nn.GroupNorm, x: torch.Tensor, silu: bool, add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``silu(norm(x + add[:, :, None, None]))`` / ``norm(...)`` -- one fused pass over a channels-last activation when the
    kernel applies (``add``: fp32 ``[B, C]``)."""
    if _enabled(norm, x) and _nhwc(x):
        gamma, beta = _f32_params(norm, "weight", "bias")
        if not torch.is_grad_enabled():
            from .. import ops
            return ops.group_norm_nhwc(x, gamma, beta, norm.num_groups, norm.eps, silu, add)
        if _frozen(norm.weight, norm.bias, add):
            return _GroupNormActFn.apply(x, add, gamma, beta, norm.num_groups, norm.eps, silu)
    if add is not None:
        x = x + add.to(x.dtype)[:, :, None, None]
    y = norm(x)
    return F.silu(y) if silu else y


class _LayerNormFn(torch.autograd.Function):
    """Training-time LayerNorm with a frozen affine: one launch forward, one for the input gradient; only x is kept."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps):
        from .. import ops
        ctx.save_for_backward(x, gamma)
        ctx.eps = eps
        return ops.layer_norm(x, gamma, beta, eps)

    @staticmethod
    def backward(ctx, dy):
        from .. import ops
        x, gamma = ctx.saved_tensors
        return ops.layer_norm_bwd(x, dy.contiguous(), gamma, ctx.eps), None, None, None


def layer_norm(norm: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
    if _enabled(norm, x) and x.is_contiguous() and x.shape[-1] % 8 == 0 and x.shape[-1] <= 1280:
        gamma, beta = _f32_params(norm, "weight", "bias")
        if not torch.is_grad_enabled():
            from .. import ops
            return ops.layer_norm(x, gamma, beta, norm.eps)
        if _frozen(norm.weight, norm.bias):
            return _LayerNormFn.apply(x, gamma, beta, norm.eps)
    return norm(x)


class AttnProcessor2_0:
    """Stock SDPA processor for the self-attention (attn1) layers -- library code, outside the hot path."""

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, **kw):
        B, S, C = hidden_states.shape
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        if isinstance(ctx, tuple):
            ctx = ctx[0]
        h = attn.heads
        q = attn.to_q(hidden_states).view(B, -1, h, C // h).transpose(1, 2)
        k = attn.to_k(ctx).view(B, -1, h, C // h).transpose(1, 2)
        v = attn.to_v(ctx).view(B, -1, h, C // h).transpose(1, 2)
        o = F.scaled_dot_product_attention(q, k, v, dropout_p=0.0, is_causal=False)
        o = o.transpose(1, 2).reshape(B, -1, C).to(q.dtype)
        return attn.to_out[1](attn.to_out[0](o))


class Attention(nn.Module):
    """The subset of diffusers' ``Attention`` that SD-1.5 uses (bias-free q/k/v, out projection with bias)."""

    def __init__(self, query_dim: int, cross_attention_dim: Optional[int] = None, heads: int = 8):
        super().__init__()
        self.heads = heads
        self.inner_dim = query_dim
        self.cross_attention_dim = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.scale = (query_dim // heads) ** -0.5
        self.to_q = nn.Linear(query_dim, query_dim, bias=False)
        self.to_k = nn.Linear(self.cross_attention_dim, query_dim, bias=False)
        self.to_v = nn.Linear(self.cross_attention_dim, query_dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(query_dim, query_dim, bias=True), nn.Dropout(0.0)])
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = None
        self.norm_encoder_hidden_states = None
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.processor = AttnProcessor2_0()

    def set_processor(self, processor):
        # nn.Module processors become sub-modules named `processor` (their weights enter unet.state_dict(),
        # reference models/modeling_utils.py:33-37)
        if isinstance(getattr(self, "processor", None), nn.Module) and not isinstance(processor, nn.Module):
            self._modules.pop("processor", None)
        self.processor = processor

    def prepare_attention_mask(self, *a, **k):
        raise NotImplementedError("attention masks are not used by SD-1.5")

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        return self.processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                              attention_mask=attention_mask, **kw)


class _GegluFn(torch.autograd.Function):
    """Training-time GEGLU product: one launch forward, one backward; only the projection is kept."""

    @staticmethod
    def forward(ctx, h):
        from .. import ops
        ctx.save_for_backward(h)
        return ops.geglu(h)

    @staticmethod
    def backward(ctx, dy):
        from .. import ops
        (h,) = ctx.saved_tensors
        return ops.geglu_bwd(h, dy.contiguous())


class GEGLU(nn.Module):
    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)

    def _packed(self):
        """The projection's weight and bias in the row order of ops.linear_geglu, refreshed when a parameter changes."""
        ps = (self.proj.weight, self.proj.bias)
        key = tuple((p.data_ptr(), p._version) for p in ps)
        cached = getattr(self, "_pv_geglu", None)
        if cached is None or cached[0] != key:
            from .. import ops
            cached = (key, ops.pack_geglu_weight(*ps))
            self._pv_geglu = cached
        return cached[1]

    def forward(self, x):
        if (_fused(self, x) and x.is_contiguous() and x.shape[-1] % 64 == 0 and self.proj.out_features % 160 == 0
                and self.proj.bias is not None):
            # inference: projection and GEGLU product in one launch; the [M, 2N] projection is never written
            from .. import ops
            return ops.linear_geglu(x, *self._packed())
        h = self.proj(x)
        if _enabled(self, h) and h.is_contiguous() and h.shape[-1] % 16 == 0:
            if torch.is_grad_enabled() and h.requires_grad:
                return _GegluFn.apply(h)
            from .. import ops
            return ops.geglu(h)
        x, gate = h.chunk(2, dim=-1)
        return x * F.gelu(gate)


class FeedForward(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.net = nn.ModuleList([GEGLU(dim, dim * 4), nn.Dropout(0.0), nn.Linear(dim * 4, dim)])

    def forward(self, x):
        for m in self.net:
            x = m(x)
        return x


class BasicTransformerBlock(nn.Module):
    def __init__(self, dim, heads, cross_attention_dim):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn1 = Attention(dim, None, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.attn2 = Attention(dim, cross_attention_dim, heads)
        self.norm3 = nn.LayerNorm(dim)
        self.ff = FeedForward(dim)

    def forward(self, x, encoder_hidden_states, cross_attention_kwargs=None):
        # diffusers passes cross_attention_kwargs (e.g. ip_adapter_masks) to both attention layers
        kw = cross_attention_kwargs or {}
        if (_fused(self.norm2, x) and _fused(self.norm3, x) and x.is_contiguous() and x.shape[-1] % 8 == 0
                and x.shape[-1] <= 1280):
            # inference: each residual sum rides in the pass of the LayerNorm that follows it
            from .. import ops
            h = self.attn1(layer_norm(self.norm1, x), **kw)
            x, n = ops.add_layer_norm(h.contiguous(), x, *_f32_params(self.norm2, "weight", "bias"), self.norm2.eps)
            h = self.attn2(n, encoder_hidden_states=encoder_hidden_states, **kw)
            x, n = ops.add_layer_norm(h.contiguous(), x, *_f32_params(self.norm3, "weight", "bias"), self.norm3.eps)
            return self.ff(n) + x
        x = self.attn1(layer_norm(self.norm1, x), **kw) + x
        x = self.attn2(layer_norm(self.norm2, x), encoder_hidden_states=encoder_hidden_states, **kw) + x
        return self.ff(layer_norm(self.norm3, x)) + x


class Transformer2DModel(nn.Module):
    def __init__(self, channels, heads, cross_attention_dim, groups=32):
        super().__init__()
        self.norm = nn.GroupNorm(groups, channels, eps=1e-6)
        self.proj_in = nn.Conv2d(channels, channels, 1)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(channels, heads, cross_attention_dim)])
        self.proj_out = nn.Conv2d(channels, channels, 1)

    def forward(self, x, encoder_hidden_states, cross_attention_kwargs=None):
        B, C, H, W = x.shape
        res = x
        if _enabled(self.norm, x) and _nhwc(x):
            # channels-last: the 1x1 convolutions are Linears on the [B, HW, C] view (bias in the GEMM epilogue instead of a
            # broadcast-add launch), the residual sum runs on the same view
            h = group_norm_act(self.norm, x, False).permute(0, 2, 3, 1).reshape(B, H * W, C)
            h = F.linear(h, self.proj_in.weight.view(C, C), self.proj_in.bias)
            for blk in self.transformer_blocks:
                h = blk(h, encoder_hidden_states, cross_attention_kwargs)
            h = F.linear(h, self.proj_out.weight.view(C, C), self.proj_out.bias)
            h = h + res.permute(0, 2, 3, 1).reshape(B, H * W, C)
            return h.reshape(B, H, W, C).permute(0, 3, 1, 2)
        h = self.proj_in(group_norm_act(self.norm, x, False))
        h = h.permute(0, 2, 3, 1).reshape(B, H * W, C)
        for blk in self.transformer_blocks:
            h = blk(h, encoder_hidden_states, cross_attention_kwargs)
        h = h.reshape(B, H, W, C).permute(0, 3, 1, 2)      # NHWC-strided view: free under channels_last
        return self.proj_out(h) + res


class ResnetBlock2D(nn.Module):
    def __init__(self, cin, cout, temb_ch, groups=32):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=1e-5)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb_ch, cout)
        self.norm2 = nn.GroupNorm(groups, cout, eps=1e-5)
        self.dropout = nn.Dropout(0.0)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None

    def forward(self, x, temb):
        if (_enabled(self.norm1, x) and _nhwc(x) and self.conv1.out_channels % 8 == 0
                and (not torch.is_grad_enabled()
                     or _frozen(temb, self.conv1.bias, self.conv2.bias, self.time_emb_proj.weight, self.time_emb_proj.bias,
                                None if self.conv_shortcut is None else self.conv_shortcut.bias))):
            # the convolutions run bias-free; conv1's bias and the time-embedding projection enter norm2's two passes as a
            # per-(sample, channel) addend, conv2's (and the shortcut's) bias enters the residual sum: 2 launches instead
            # of 4 broadcast adds that each re-read and re-write the activation
            c1, c2, cs = self.conv1, self.conv2, self.conv_shortcut
            h = F.conv2d(group_norm_act(self.norm1, x, True), c1.weight, None, c1.stride, c1.padding)
            add = self.time_emb_proj(F.silu(temb)).float() + _f32_params(c1, "bias")[0]
            h = F.conv2d(group_norm_act(self.norm2, h, True, add), c2.weight, None, c2.stride, c2.padding)
            bias = _f32_params(c2, "bias")[0]
            if cs is not None:
                x = F.conv2d(x, cs.weight, None, cs.stride, cs.padding)
                bias = self._shortcut_bias()
            if torch.is_grad_enabled() and (x.requires_grad or h.requires_grad):
                return _AddBiasFn.apply(x, h, bias)
            from .. import ops
            return ops.add_bias_nhwc(x, h, bias)
        h = self.conv1(group_norm_act(self.norm1, x, True))
        h = h + self.time_emb_proj(F.silu(temb))[:, :, None, None]
        h = self.conv2(self.dropout(group_norm_act(self.norm2, h, True)))
        if self.conv_shortcut is not None:
            x = self.conv_shortcut(x)
        return x + h


def _resnet_shortcut_bias(self):
    """conv2.bias + conv_shortcut.bias in fp32 (cached by parameter versions)."""
    c2, cs = self.conv2, self.conv_shortcut
    key = (c2.bias.data_ptr(), c2.bias._version, cs.bias.data_ptr(), cs.bias._version)
    cached = getattr(self, "_pv_sum_bias", None)
    if cached is None or cached[0] != key:
        cached = (key, (c2.bias.detach().float() + cs.bias.detach().float()).contiguous())
        self._pv_sum_bias = cached
    return cached[1]


ResnetBlock2D._shortcut_bias = _resnet_shortcut_bias


class Downsample2D(nn.Module):
    def __init__(self, ch):
        super().__init__()
        self.conv = nn.Conv2d(ch, ch, 3, stride=2, padding=1)

    def forward(self, x):
        return self.conv(x)


class Upsample2D(nn.Module):
    def __init__(self, ch):
        super().__init__()
        self.conv = nn.Conv2d(ch, ch, 3, padding=1)

    def forward(self, x):
        return self.conv(F.interpolate(x, scale_factor=2.0, mode="nearest"))


class DownBlock(nn.Module):
    def __init__(self, cin, cout, temb_ch, layers, heads, cross_dim, has_attn, add_down):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(cin if i == 0 else cout, cout, temb_ch) for i in range(layers)])
        self.attentions = nn.ModuleList(
            [Transformer2DModel(cout, heads, cross_dim) for _ in range(layers)]) if has_attn else None
        self.downsamplers = nn.ModuleList([Downsample2D(cout)]) if add_down else None

    def forward(self, x, temb, ctx, cross_attention_kwargs=None):
        outs = []
        for i, r in enumerate(self.resnets):
            x = r(x, temb)
            if self.attentions is not None:
                x = self.attentions[i](x, ctx, cross_attention_kwargs)
            outs.append(x)
        if self.downsamplers is not None:
            x = self.downsamplers[0](x)
            outs.append(x)
        return x, outs


class UpBlock(nn.Module):
    def __init__(self, cin, cout, prev_out, temb_ch, layers, heads, cross_dim, has_attn, add_up):
        super().__init__()
        res = []
        for i in range(layers):
            skip = cin if i == layers - 1 else cout
            rin = prev_out if i == 0 else cout
            res.append(ResnetBlock2D(rin + skip, cout, temb_ch))
        self.resnets = nn.ModuleList(res)
        self.attentions = nn.ModuleList(
            [Transformer2DModel(cout, heads, cross_dim) for _ in range(layers)]) if has_attn else None
        self.upsamplers = nn.ModuleList([Upsample2D(cout)]) if add_up else None

    def forward(self, x, skips, temb, ctx, cross_attention_kwargs=None):
        for i, r in enumerate(self.resnets):
            x = torch.cat([x, skips.pop()], dim=1)
            x = r(x, temb)
            if self.attentions is not None:
                x = self.attentions[i](x, ctx, cross_attention_kwargs)
        if self.upsamplers is not None:
            x = self.upsamplers[0](x)
        return x


class MidBlock(nn.Module):
    def __init__(self, ch, temb_ch, heads, cross_dim):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2D(ch, ch, temb_ch), ResnetBlock2D(ch, ch, temb_ch)])
        self.attentions = nn.ModuleList([Transformer2DModel(ch, heads, cross_dim)])

    def forward(self, x, temb, ctx, cross_attention_kwargs=None):
        x = self.resnets[0](x, temb)
        x = self.attentions[0](x, ctx, cross_attention_kwargs)
        return self.resnets[1](x, temb)


class TimestepEmbedding(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.linear_1 = nn.Linear(cin, cout)
        self.linear_2 = nn.Linear(cout, cout)

    def forward(self, x):
        return self.linear_2(F.silu(self.linear_1(x)))


def timestep_sinusoid(t: torch.Tensor, dim: int) -> torch.Tensor:
    """diffusers ``Timesteps(dim, flip_sin_to_cos=True, downscale_freq_shift=0)``."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    args = t.float()[:, None] * freqs[None]
    return torch.cat([torch.cos(args), torch.sin(args)], dim=-1)


class UNetSD15(nn.Module):
    """SD-1.5 defaults: block_out_channels=(320,640,1280,1280), layers_per_block=2, 8 heads, cross dim 768,
    cross-attention in the first three down blocks / last three up blocks / the mid block -> 16 attn2 layers."""

    def __init__(self, in_channels=4, out_channels=4, block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280),
                 layers_per_block=2, heads=8, cross_attention_dim=768, sample_size=64):
        super().__init__()
        boc = tuple(block_out_channels)
        n = len(boc)
        self.config = SimpleNamespace(in_channels=in_channels, out_channels=out_channels, block_out_channels=boc,
                                      layers_per_block=layers_per_block, attention_head_dim=heads,
                                      cross_attention_dim=cross_attention_dim, sample_size=sample_size)
        temb_ch = boc[0] * 4
        self.conv_in = nn.Conv2d(in_channels, boc[0], 3, padding=1)
        self.time_embedding = TimestepEmbedding(boc[0], temb_ch)
        self.down_blocks = nn.ModuleList()
        cout = boc[0]
        for i in range(n):
            cin, cout = cout, boc[i]
            last = i == n - 1
            self.down_blocks.append(DownBlock(cin, cout, temb_ch, layers_per_block, heads, cross_attention_dim,
                                              has_attn=not last or n == 1, add_down=not last))
        self.mid_block = MidBlock(boc[-1], temb_ch, heads, cross_attention_dim)
        self.up_blocks = nn.ModuleList()
        rev = list(reversed(boc))
        cout = rev[0]
        for i in range(n):
            prev_out, cout = cout, rev[i]
            cin = rev[min(i + 1, n - 1)]
            last = i == n - 1
            self.up_blocks.append(UpBlock(cin, cout, prev_out, temb_ch, layers_per_block + 1, heads,
                                          cross_attention_dim, has_attn=i > 0 or n == 1, add_up=not last))
        self.conv_norm_out = nn.GroupNorm(32, boc[0], eps=1e-5)
        self.conv_out = nn.Conv2d(boc[0], out_channels, 3, padding=1)

    # ---- diffusers attention-processor protocol ------------------------------------------------
    @property
    def attn_processors(self) -> Dict[str, object]:
        procs = {}
        for name, m in self.named_modules():
            if isinstance(m, Attention):
                procs[f"{name}.processor"] = m.processor
        return procs

    def set_attn_processor(self, processor):
        mods = {f"{name}.processor": m for name, m in self.named_modules() if isinstance(m, Attention)}
        if isinstance(processor, dict):
            if len(processor) != len(mods):
                raise ValueError(f"A dict of processors was passed, but the number of processors {len(processor)} "
                                 f"does not match the number of attention layers: {len(mods)}.")
            for k, m in mods.items():
                m.set_processor(processor[k])
        else:
            for m in mods.values():
                m.set_processor(processor)

    def set_fused_epilogues(self, enabled: bool):
        """photoverse_b200 epilogue kernels (GroupNorm + SiLU, LayerNorm, GEGLU, bias / residual sums) for this model's
        inference passes (default on) or the stock PyTorch ops."""
        for m in self.modules():
            if isinstance(m, (nn.GroupNorm, nn.LayerNorm, GEGLU)):
                m._pv_fused = bool(enabled)
        return self

    def forward(self, sample, timestep, encoder_hidden_states, cross_attention_kwargs=None):
        """``cross_attention_kwargs``: extra keyword arguments of every attention processor call, as diffusers'
        ``UNet2DConditionModel`` passes them (e.g. ``{"ip_adapter_masks": [mask]}``)."""
        if not torch.is_tensor(timestep):
            timestep = torch.tensor([timestep], device=sample.device)
        t = timestep.reshape(-1).expand(sample.shape[0]) if timestep.numel() == 1 else timestep
        temb = self.time_embedding(timestep_sinusoid(t, self.config.block_out_channels[0]).to(sample.dtype))
        x = self.conv_in(sample)
        skips = [x]
        for blk in self.down_blocks:
            x, outs = blk(x, temb, encoder_hidden_states, cross_attention_kwargs)
            skips += outs
        x = self.mid_block(x, temb, encoder_hidden_states, cross_attention_kwargs)
        for blk in self.up_blocks:
            x = blk(x, skips, temb, encoder_hidden_states, cross_attention_kwargs)
        x = self.conv_out(group_norm_act(self.conv_norm_out, x, True))
        return SimpleNamespace(sample=x)
