"""One PhotoVerse training step around the B200 path (counterpart of reference train.py:463-549, BASELINE config 4).

Scope: the caller of the path.  VAE, CLIP encoders and the tokenizer are outside it (SURVEY §2): their outputs -- noisy
latents, timesteps, CLIP ViT-L/14 hidden states, text-encoder states -- are the inputs here (synthetic in the bench).
What it keeps from the reference:
  :495,502  text_adapter / image_adapter over all 5 token heads (no token_index)
  :505      noise_pred = unet(noisy, t, encoder_hidden_states=(text, image_tokens))  -- 16 processors in grad mode:
            stochastic fusion rule, one torch.rand(1) per layer (attention_processor.py:411-420)
  :509      L_text = mean |concept_text_embeddings|         :512-513  L_vis = mean ||V_ip|| over the 16 layers
  :516      L_mse  = MSE(noise_pred, noise)                 :535      loss = L_mse + 0.01 L_text + 0.001 L_vis
  :538      backward through the frozen UNet into the trainable set
  :541-544  clip_grad_norm_(1.0) per module group           :547      AdamW
  :497-499  encoder_hidden_states = text_encoder({ids, concept_text_embeddings, concept_placeholder_idx})[0]: the text
            adapter's concept embeddings replace the placeholder token inside the (frozen) CLIP text tower
            (models/clip.py:17-24, 50-63 -> host/text_encoder.py + pv_inject_concept_fwd/_bwd), so the denoising loss
            reaches the text adapter through the text branch of all 16 processors, as in the reference
Data parallel: gradients are allreduced as bucketed slices of one flat buffer, launched under the backward pass
(photoverse_b200.host.parallel).  Without a ``text_encoder`` the step takes ``batch.text`` as a plain input (the text
adapter is then trained by L_text alone -- the round-1 behaviour, kept for the kernels' unit tests).
"""
import contextlib
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.nn.functional as F

from ..autograd import convert
from ..loss import train_loss
from ..unet import get_visual_cross_attention_values_norm
from .parallel import FlatGradBuffer, OverlappedGradReducer, trainable_named_parameters


@dataclass
class TrainBatch:
    noisy_latents: torch.Tensor        # [B,4,h,w]
    timesteps: torch.Tensor            # [B] float
    noise: torch.Tensor                # [B,4,h,w] regression target (epsilon prediction)
    clip_hidden: List[torch.Tensor]    # 5 x [B,257,1024]
    text: torch.Tensor                 # [B,77,768]   (used only when the Trainer has no text encoder)
    text_ids: Optional[torch.Tensor] = None          # [B,77] int64 prompt token ids
    placeholder_idx: Optional[List[int]] = None      # B positions of the concept placeholder (datasets/utils.py:215-220)


def synthetic_train_batch(batch: int, latent: int = 64, seed: int = 0, device="cpu", dtype=torch.float32) -> TrainBatch:
    g = torch.Generator().manual_seed(seed)

    def rn(*shape):
        return torch.randn(*shape, generator=g, dtype=torch.float32).to(device=device, dtype=dtype)
    t = torch.randint(0, 1000, (batch,), generator=g).to(device=device, dtype=torch.float32)
    b = TrainBatch(rn(batch, 4, latent, latent), t, rn(batch, 4, latent, latent), [rn(batch, 257, 1024) for _ in range(5)],
                   rn(batch, 77, 768))
    b.text_ids = torch.randint(0, 49408, (batch, 77), generator=g).to(device)
    b.placeholder_idx = [int(v) for v in torch.randint(1, 20, (batch,), generator=g)]   # "a photo of S" style prompts
    return b


class Trainer:
    """Persistent state of the training loop: trainable set, flat gradient buffer, AdamW."""

    GROUPS = ("text_adapter.", "image_adapter.", "unet.")

    def __init__(self, unet, image_adapter, text_adapter, lr: float = 1e-4, weight_decay: float = 1e-2, group=None,
                 text_encoder=None, autocast_dtype: Optional[torch.dtype] = None):
        """``autocast_dtype=torch.bfloat16``: the forward pass runs under ``torch.autocast("cuda", torch.bfloat16)``, the
        reference's ``accelerate --mixed_precision bf16`` over float32 weights (DESIGN.md 4.9); float16 is refused, the
        path has no fp16 backward."""
        if autocast_dtype not in (None, torch.bfloat16):
            raise ValueError(f"autocast_dtype must be None or torch.bfloat16 (training has no float16 backward), got "
                             f"{autocast_dtype}")
        self.autocast_dtype = autocast_dtype
        self.unet, self.image_adapter, self.text_adapter = unet, image_adapter, text_adapter
        self.text_encoder = text_encoder             # frozen CLIP text tower with concept injection (host/text_encoder.py)
        self.named = trainable_named_parameters(unet, image_adapter, text_adapter)
        if not self.named:
            raise ValueError("nothing to train: no parameter of the adapters / unet requires grad")
        self.buf = FlatGradBuffer(self.named)
        self.opt = torch.optim.AdamW([p for _, p in self.named], lr=lr, betas=(0.9, 0.999), weight_decay=weight_decay,
                                     eps=1e-8)          # train.py:94-107 defaults
        self.group = group
        self.reducer = OverlappedGradReducer(self.buf, group)      # bucketed allreduce under the backward pass (world > 1)
        self.buckets_overlapped = 0

    def loss(self, b: TrainBatch):
        concept = self.text_adapter(b.clip_hidden)                                    # train.py:495
        if self.text_encoder is not None:                                             # train.py:497-499
            text = self.text_encoder({"text_input_ids": b.text_ids, "concept_text_embeddings": concept.to(b.text.dtype),
                                      "concept_placeholder_idx": b.placeholder_idx})[0]
        else:
            text = b.text
        img_tokens = self.image_adapter(b.clip_hidden)                                # train.py:502
        pred = self.unet(b.noisy_latents, b.timesteps, encoder_hidden_states=(text, img_tokens)).sample     # :505
        vnorms = get_visual_cross_attention_values_norm(self.unet)                    # :512 (stack of the 16 side outputs)
        if pred.is_cuda:      # :509-535 in one reduction kernel (+ one backward kernel): photoverse_b200.loss
            if self.autocast_dtype is not None:     # :516 mse_loss(pred.float(), target.float()): the target is not rounded
                pred = pred if pred.dtype == torch.float32 else convert(pred, torch.float32)
                return train_loss(pred, b.noise.float(), concept, vnorms, 0.01, 0.001)
            return train_loss(pred, b.noise, concept, vnorms, 0.01, 0.001)
        l_text = concept.float().abs().mean()                                         # :509
        l_vis = vnorms.float().mean()                                                 # :513
        l_mse = F.mse_loss(pred.float(), b.noise.float(), reduction="mean")           # :516
        return l_mse + 0.01 * l_text + 0.001 * l_vis, (l_mse, l_text, l_vis)          # :535

    def expected_gradients(self) -> List[bool]:
        """Which trainable parameters take part in this step's graph: the fusion rule drawn in the forward pass
        (``last_fusion`` of every attn2 processor) drops ``to_k_ip`` of an image-less layer and the K/V LoRA factors of
        a text-less one (attention_processor.py:413-418); everything else receives a gradient."""
        from ..attention_processor import PhotoVerseAttnProcessor2_0
        off = []
        for name, module in self.unet.named_modules():
            proc = getattr(module, "processor", None)
            if isinstance(proc, PhotoVerseAttnProcessor2_0):
                w_text, w_img = proc.last_fusion
                if w_img == 0.0:
                    off.append(f"unet.{name}.processor.to_k_ip.")
                if w_text == 0.0:
                    off += [f"unet.{name}.to_k.lora_", f"unet.{name}.to_v.lora_"]
        return [not any(n.startswith(pre) for pre in off) for n, _ in self.named]

    def step(self, b: TrainBatch, max_grad_norm: float = 1.0):
        self.opt.zero_grad(set_to_none=True)
        autocast = (contextlib.nullcontext() if self.autocast_dtype is None
                    else torch.autocast("cuda", dtype=self.autocast_dtype))
        with torch.enable_grad(), autocast:
            loss, parts = self.loss(b)
        self.reducer.begin(self.expected_gradients())
        loss.backward()                                                               # :538
        ev = getattr(self, "reducer_events", None)        # bench: the exposed (not overlapped) part of the allreduce
        if ev is not None:
            ev[0].record()
        self.buckets_overlapped = self.reducer.finish()                               # mean over ranks in the flat buffer
        if ev is not None:
            ev[1].record()
            self.reducer_events = None
        self.buf.clip_groups_(self.GROUPS, max_grad_norm)                             # :541-544
        self.buf.unpack()
        self.opt.step()                                                               # :547
        return loss.detach(), tuple(p.detach() for p in parts)
