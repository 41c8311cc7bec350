"""Generation loop around the hot path (counterpart of the reference's ``models/infer.py:run_inference``).

Scope note: this is the *caller* of the B200 path (SURVEY.md §8 f1), written in plain PyTorch.  CLIP encoders, the
tokenizer and the VAE are outside the path (SURVEY §2) -- their outputs (CLIP ViT-L/14 hidden states, text-encoder
states, initial noise) are the inputs here, and the final latents are the output.

What it keeps from the reference (infer.py):
  :89-91   text_adapter / image_adapter (cond and zero-image "uncond") run once per generation, token_index=0 default
  :98-119  per step: eps_uncond and eps_cond from the UNet with (text, image) conditioning tuples, classifier-free
           guidance combine, scheduler step
What it does the B200 way:
  * the two UNet calls of a step are ONE doubled-batch call (mode "batched"); "two_call" reproduces the reference's
    call pattern exactly; "cond_only" skips the uncond branch, valid only for guidance_scale == 1
  * K/V projections of all 16 attn2 layers are computed once per generation and cached (SURVEY §0.1 D7)
  * one UNet evaluation is captured in a CUDA graph and replayed for the remaining steps (no host sync in the loop)
  * DDIM (BASELINE.json) instead of DPM-Solver++ -- same scheduler on both arms of every comparison
"""
import contextlib
from dataclasses import dataclass
from typing import List, Optional

import torch

from .. import _lib
from ..attention_processor import release_mask_rows
from ..unet import prepare_kv, set_kv_cache
from .ddim import make_ddim_schedule
from .dpm_solver import make_dpmpp_2m_schedule


@dataclass
class GenInputs:
    clip_hidden: List[torch.Tensor]           # T x [B,257,1024]: [last_hidden_state, hs[4], hs[8], hs[12], hs[16]]
    clip_hidden_uncond: List[torch.Tensor]    # same for the all-zero image (infer.py:77-78)
    text: torch.Tensor                        # [B,77,768] text-encoder states (concept tokens injected upstream)
    text_uncond: torch.Tensor                 # [B,77,768] for the empty prompt
    noise: torch.Tensor                       # [B,4,h,w]

    def to(self, device=None, dtype=None, non_blocking=False):
        def cv(t):
            return t.to(device=device, dtype=dtype, non_blocking=non_blocking)
        return GenInputs([cv(t) for t in self.clip_hidden], [cv(t) for t in self.clip_hidden_uncond],
                         cv(self.text), cv(self.text_uncond), cv(self.noise))

    def nbytes(self) -> int:
        ts = self.clip_hidden + self.clip_hidden_uncond + [self.text, self.text_uncond, self.noise]
        return sum(t.numel() * t.element_size() for t in ts)


class _GraphedUNet:
    """One UNet evaluation captured in a CUDA graph (static input buffers, replayed every step)."""

    def __init__(self, unet, latent_shape, ctx, dtype, device, cak=None):
        self.unet = unet
        self.ctx = ctx
        self.x = torch.zeros(latent_shape, device=device, dtype=dtype)
        self.t = torch.zeros(1, device=device, dtype=torch.float32)
        s = torch.cuda.Stream(device=device)
        s.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(s):
            for _ in range(2):       # warm-up outside capture: packs weights, fills the K/V (and mask) caches, cuDNN autotune
                unet(self.x, self.t, encoder_hidden_states=ctx, cross_attention_kwargs=cak)
        torch.cuda.current_stream(device).wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = unet(self.x, self.t, encoder_hidden_states=ctx, cross_attention_kwargs=cak).sample

    def __call__(self, x, t_dev):
        self.x.copy_(x)
        self.t.copy_(t_dev)
        self.graph.replay()
        return self.out


def _autocast(dtype: Optional[torch.dtype]):
    """``torch.autocast("cuda", dtype)`` for a float32 model run in mixed precision; None leaves the caller's autocast state
    as it is.  Autocast's weight-cast cache stays off: cast weights cached inside a CUDA-graph capture would be freed when
    the region exits."""
    if dtype is None:
        return contextlib.nullcontext()
    return torch.autocast("cuda", dtype=dtype, cache_enabled=False)


@torch.no_grad()
def run_generation(unet, image_adapter, text_adapter, inputs: GenInputs, num_steps: int = 50,
                   guidance_scale: float = 1.0, token_index=0, mode: str = "batched", use_cuda_graph: bool = True,
                   kv_cache: bool = True, return_aux: bool = False, scheduler: str = "ddim",
                   autocast_dtype: Optional[torch.dtype] = None, ip_adapter_masks=None):
    """Returns the final latents [B,4,h,w] (and the adapter outputs if ``return_aux``).  ``autocast_dtype``: run the
    adapters and every UNet evaluation (warm-up, graph capture and replay) under ``torch.autocast("cuda", autocast_dtype)``
    -- a float32 model in the reference's mixed precision.  ``ip_adapter_masks``: diffusers' regional identity masks
    (a list with one [1 or B, 1, H, W] tensor), passed to every UNet evaluation as ``cross_attention_kwargs``; with
    batched CFG a mask of batch B is repeated for the unconditional half, as the diffusers pipeline does."""
    with _autocast(autocast_dtype):
        return _run_generation(unet, image_adapter, text_adapter, inputs, num_steps, guidance_scale, token_index, mode,
                               use_cuda_graph, kv_cache, return_aux, scheduler, ip_adapter_masks)


def _mask_kwargs(ip_adapter_masks, batched: bool):
    """``cross_attention_kwargs`` of the UNet evaluations: with batched CFG the rows are [uncond | cond], so a mask of
    batch B > 1 is concatenated with itself (a mask of batch 1 broadcasts already)."""
    if ip_adapter_masks is None:
        return None
    masks = list(ip_adapter_masks.unsqueeze(1)) if isinstance(ip_adapter_masks, torch.Tensor) else list(ip_adapter_masks)
    if batched:
        masks = [m if (not isinstance(m, torch.Tensor) or m.shape[0] == 1) else torch.cat([m, m]) for m in masks]
    return {"ip_adapter_masks": masks}


def _run_generation(unet, image_adapter, text_adapter, inputs, num_steps, guidance_scale, token_index, mode,
                    use_cuda_graph, kv_cache, return_aux, scheduler, ip_adapter_masks=None):
    assert mode in ("batched", "two_call", "cond_only")
    if mode == "cond_only" and guidance_scale != 1.0:
        raise ValueError("mode='cond_only' drops the unconditional branch: only valid for guidance_scale == 1")
    dev, dtype = inputs.noise.device, inputs.noise.dtype
    assert scheduler in ("ddim", "dpmpp_2m")          # ddim: BASELINE metric; dpmpp_2m: the reference's sampler (infer.py:39-40)
    sched = make_ddim_schedule(num_steps) if scheduler == "ddim" else make_dpmpp_2m_schedule(num_steps)
    x0_prev = None

    # ---- adapters: once per generation (infer.py:89-91) ----
    concept_text = text_adapter(inputs.clip_hidden, token_index=token_index) if text_adapter is not None else None
    img_tokens = image_adapter(inputs.clip_hidden, token_index=token_index)
    img_tokens_uncond = image_adapter(inputs.clip_hidden_uncond, token_index=token_index)

    latents = inputs.noise * sched.init_noise_sigma
    B = latents.shape[0]
    if mode == "batched":
        ctx = (torch.cat([inputs.text_uncond, inputs.text]).contiguous(),
               torch.cat([img_tokens_uncond, img_tokens]).contiguous())
        ctxs = [ctx]
    elif mode == "two_call":
        ctxs = [(inputs.text_uncond.contiguous(), img_tokens_uncond.contiguous()),
                (inputs.text.contiguous(), img_tokens.contiguous())]
    else:
        ctxs = [(inputs.text.contiguous(), img_tokens.contiguous())]

    cak = _mask_kwargs(ip_adapter_masks, mode == "batched")
    set_kv_cache(unet, kv_cache)
    ts_dev = torch.tensor(sched.timesteps, device=dev, dtype=torch.float32)
    rows = 2 * B if mode == "batched" else B
    lat_shape = (rows,) + tuple(latents.shape[1:])
    evals = None
    if use_cuda_graph and dev.type == "cuda":
        evals = [_GraphedUNet(unet, lat_shape, c, dtype, dev, cak) for c in ctxs]
    try:
        for i in range(num_steps):
            t_dev = ts_dev[i:i + 1]
            x_in = torch.cat([latents, latents]) if mode == "batched" else latents
            outs = []
            for j, c in enumerate(ctxs):
                if evals is not None:
                    outs.append(evals[j](x_in, t_dev))
                else:
                    outs.append(unet(x_in, t_dev, encoder_hidden_states=c, cross_attention_kwargs=cak).sample)
            if mode == "batched":
                eps_u, eps_c = outs[0].chunk(2)
            elif mode == "two_call":
                eps_u, eps_c = outs
            else:
                eps_u = eps_c = outs[0]
            if mode == "cond_only":
                eps = eps_c
            else:
                eps = eps_u + guidance_scale * (eps_c - eps_u)          # infer.py:116
            if scheduler == "ddim":
                latents = sched.c_x[i] * latents + sched.c_eps[i] * eps     # DDIM step (eta = 0)
            else:                                                            # DPM-Solver++(2M), data-prediction form
                x0 = sched.kx[i] * latents + sched.ke[i] * eps
                nxt = sched.cx[i] * latents + sched.c0[i] * x0
                if sched.c0p[i] != 0.0:
                    nxt = nxt + sched.c0p[i] * x0_prev
                latents, x0_prev = nxt, x0
    finally:
        set_kv_cache(unet, False)
    if return_aux:
        return latents, {"concept_text": concept_text, "img_tokens": img_tokens, "img_tokens_uncond": img_tokens_uncond}
    return latents


def synthetic_inputs(batch: int, latent: int = 64, tokens: int = 257, T: int = 5, seed: int = 0,
                     device="cpu", dtype=torch.float32, pin: bool = False) -> GenInputs:
    """Synthetic stand-ins for the encoder outputs (there is no network for real weights / images):
    N(0,1) CLIP hidden states, text states and noise; the "uncond" image is a different fixed draw."""
    g = torch.Generator().manual_seed(seed)

    def rn(*shape):
        t = torch.randn(*shape, generator=g, dtype=torch.float32).to(dtype)
        if pin and torch.cuda.is_available():
            t = t.pin_memory()
        return t.to(device) if str(device) != "cpu" else t

    clip = [rn(batch, tokens, 1024) for _ in range(T)]
    clip_u = [rn(1, tokens, 1024).expand(batch, tokens, 1024).contiguous() for _ in range(T)]
    if pin and torch.cuda.is_available() and str(device) == "cpu":
        clip_u = [t.pin_memory() for t in clip_u]
    return GenInputs(clip, clip_u, rn(batch, 77, 768), rn(1, 77, 768).expand(batch, 77, 768).contiguous(),
                     rn(batch, 4, latent, latent))


class GenerationEngine:
    """Persistent generation state for repeated generations of one geometry (bench / serving loop):
    static device buffers for the encoder outputs, statically addressed K/V caches refreshed once per generation,
    and ONE captured CUDA graph of the UNet evaluation that every step of every generation replays.
    ``generate()`` performs no host<->device synchronisation."""

    def __init__(self, unet, image_adapter, text_adapter, batch: int, latent: int = 64, num_steps: int = 50,
                 guidance_scale: float = 1.0, token_index=0, mode: str = "batched", dtype=torch.bfloat16,
                 device="cuda", num_heads_T: int = 5, use_cuda_graph: bool = True,
                 autocast_dtype: Optional[torch.dtype] = None, ip_mask_shape=None):
        """``dtype``: the model's and the encoder buffers' dtype; ``autocast_dtype``: run the adapters and the UNet
        evaluations (warm-up, capture, replay) under ``torch.autocast("cuda", autocast_dtype)`` (None: off).
        ``ip_mask_shape`` (H, W): every generation applies a regional identity mask (diffusers' ``ip_adapter_masks``) of
        that size, a static fp32 input set by :meth:`load_inputs`; it is downsampled inside the captured evaluation."""
        assert mode in ("batched", "two_call", "cond_only")
        if mode == "cond_only" and guidance_scale != 1.0:
            raise ValueError("mode='cond_only' is only valid for guidance_scale == 1")
        self.unet, self.image_adapter, self.text_adapter = unet, image_adapter, text_adapter
        self.B, self.latent, self.num_steps, self.g = batch, latent, num_steps, float(guidance_scale)
        self.token_index, self.mode, self.dtype, self.dev = token_index, mode, dtype, torch.device(device)
        self.use_graph = use_cuda_graph
        self.autocast_dtype = autocast_dtype
        self.sched = make_ddim_schedule(num_steps)
        self.ts_dev = torch.tensor(self.sched.timesteps, device=self.dev, dtype=torch.float32)
        self.inp = synthetic_inputs(batch, latent, T=num_heads_T, seed=0, device=self.dev, dtype=dtype)
        Li = 1 if (token_index is not None and token_index != "full") else num_heads_T
        rows = 2 * batch if mode == "batched" else batch
        nctx = 2 if mode == "two_call" else 1
        self.ctx = [(torch.zeros(rows, 77, 768, device=self.dev, dtype=dtype),
                     torch.zeros(rows, Li, 768, device=self.dev, dtype=dtype)) for _ in range(nctx)]
        self.x_in = torch.zeros(rows, 4, latent, latent, device=self.dev, dtype=dtype)
        self.t_in = torch.zeros(1, device=self.dev, dtype=torch.float32)
        self.graphs = None
        self.outs = None
        self.launches_per_eval = 0      # native kernels inside one captured UNet evaluation
        self.replays = 0
        self.ip_mask = None
        if ip_mask_shape is not None:
            self.ip_mask = torch.ones(1, 1, *ip_mask_shape, device=self.dev, dtype=torch.float32)
        self._mask_rows = []
        set_kv_cache(unet, True, static=True)

    def load_inputs(self, host_inputs: GenInputs, ip_mask: Optional[torch.Tensor] = None):
        """Host (pinned) -> static device buffers; asynchronous on the current stream.  ``ip_mask`` [1, 1, H, W]: the
        regional identity mask of the following generations (engines built with ``ip_mask_shape`` only)."""
        for dst, src in zip(self.inp.clip_hidden + self.inp.clip_hidden_uncond + [self.inp.text, self.inp.text_uncond, self.inp.noise],
                            host_inputs.clip_hidden + host_inputs.clip_hidden_uncond
                            + [host_inputs.text, host_inputs.text_uncond, host_inputs.noise]):
            dst.copy_(src, non_blocking=True)
        if ip_mask is not None:
            if self.ip_mask is None:
                raise ValueError("this GenerationEngine was built without ip_mask_shape")
            self.ip_mask.copy_(ip_mask.reshape(self.ip_mask.shape), non_blocking=True)

    def _eval(self, j):
        cak = None if self.ip_mask is None else {"ip_adapter_masks": [self.ip_mask]}
        return self.unet(self.x_in, self.t_in, encoder_hidden_states=self.ctx[j], cross_attention_kwargs=cak).sample

    def _build_graphs(self):
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            for _ in range(2):
                for j in range(len(self.ctx)):
                    self._eval(j)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        self.graphs, self.outs = [], []
        for j in range(len(self.ctx)):
            g = torch.cuda.CUDAGraph()
            if self.ip_mask is not None:      # the capture downsamples the static mask: every replay sees its contents
                release_mask_rows(self.ip_mask)
            n0 = _lib.launch_count()
            with torch.cuda.graph(g):
                out = self._eval(j)
            if self.ip_mask is not None:
                self._mask_rows += release_mask_rows(self.ip_mask)      # the graph's row buffers, kept alive here
            self.launches_per_eval = _lib.launch_count() - n0
            self.graphs.append(g)
            self.outs.append(out)

    @torch.no_grad()
    def generate(self) -> torch.Tensor:
        with _autocast(self.autocast_dtype):
            return self._generate()

    def _generate(self) -> torch.Tensor:
        inp, B = self.inp, self.B
        # adapters once per generation (infer.py:89-91)
        if self.text_adapter is not None:
            self.concept_text = self.text_adapter(inp.clip_hidden, token_index=self.token_index)
        img = self.image_adapter(inp.clip_hidden, token_index=self.token_index)
        img_u = self.image_adapter(inp.clip_hidden_uncond, token_index=self.token_index)
        if self.mode == "batched":
            self.ctx[0][0][:B].copy_(inp.text_uncond); self.ctx[0][0][B:].copy_(inp.text)
            self.ctx[0][1][:B].copy_(img_u); self.ctx[0][1][B:].copy_(img)
        elif self.mode == "two_call":
            self.ctx[0][0].copy_(inp.text_uncond); self.ctx[0][1].copy_(img_u)
            self.ctx[1][0].copy_(inp.text); self.ctx[1][1].copy_(img)
        else:
            self.ctx[0][0].copy_(inp.text); self.ctx[0][1].copy_(img)
        for c in self.ctx:
            prepare_kv(self.unet, c[0], c[1])
        if self.use_graph and self.graphs is None:
            self._build_graphs()
        latents = inp.noise * self.sched.init_noise_sigma
        for i in range(self.num_steps):
            self.t_in.copy_(self.ts_dev[i:i + 1])
            if self.mode == "batched":
                self.x_in[:B].copy_(latents); self.x_in[B:].copy_(latents)
            else:
                self.x_in.copy_(latents)
            outs = []
            for j in range(len(self.ctx)):
                if self.use_graph:
                    self.graphs[j].replay()
                    self.replays += 1
                    outs.append(self.outs[j])
                else:
                    outs.append(self._eval(j))
            if self.mode == "batched":
                eps_u, eps_c = outs[0][:B], outs[0][B:]
                eps = eps_u + self.g * (eps_c - eps_u)
            elif self.mode == "two_call":
                eps = outs[0] + self.g * (outs[1] - outs[0])
            else:
                eps = outs[0]
            latents = self.sched.c_x[i] * latents + self.sched.c_eps[i] * eps
        return latents

    def close(self):
        set_kv_cache(self.unet, False)
        self.graphs = None
