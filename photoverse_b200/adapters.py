"""B200-native drop-in for the reference's ``models/adapters.py`` (PhotoVerseAdapter).

Same constructor, same ``forward(embs, token_index=None)`` contract and the same parameter names
(``mapping_{i}`` / ``mapping_patch_{i}`` = nn.Sequential with parameters at indices 0,1,3,4,6; adapters.py:13-28),
so reference checkpoints load with ``load_state_dict`` unchanged (models/modeling_utils.py:19-22).

Execution plan per call (all T selected token heads in the same launches, batched over heads):
    patches [T, B*256, 1024] --GEMM+bias--> fp32 --LN+LeakyReLU--> bf16 --GEMM+bias--> fp32 --LN+LeakyReLU--> bf16
            (float16 embeddings, inference only: fp16 wherever this plan says bf16; float32 embeddings under CUDA
             autocast: converted to the autocast dtype first, DESIGN.md 4.9)
            --mean over the 256 patches-->  cat[:, :, 1024:2048]
    cls     [T, B,     1024] --same two layers-->                            cat[:, :,    0:1024]
    out[b, t, :] = cat[t, b, :] @ [W3_cls | W3_patch]^T + (b3_cls + b3_patch)            (one K=2048 GEMM)
The patch mean is commuted in front of the last Linear (mean(L3(h)) == L3(mean(h)); SURVEY.md §2.2 A8), which
removes 256x of that layer's work; GEMMs are tcgen05 kernels, LN/LeakyReLU and the mean are vectorised
warp-shuffle kernels (photoverse_b200/csrc/pv_adapter.cu).
"""
from typing import List, Optional, Union

import torch
from torch import nn

from . import ops
from .attention_processor import _F16_TRAINING, _cast

LN_EPS = 1e-5
LRELU_SLOPE = 0.01
HIDDEN = 1024


class PhotoVerseAdapter(nn.Module):
    def __init__(self, clip_embedding_dim=1024, cross_attention_dim=768, num_tokens=5):
        super().__init__()
        self.clip_embedding_dim = clip_embedding_dim
        self.cross_attention_dim = cross_attention_dim
        self.num_tokens = num_tokens
        for i in range(num_tokens):
            for name in (f"mapping_{i}", f"mapping_patch_{i}"):
                setattr(self, name, nn.Sequential(
                    nn.Linear(clip_embedding_dim, HIDDEN), nn.LayerNorm(HIDDEN), nn.LeakyReLU(),
                    nn.Linear(HIDDEN, HIDDEN), nn.LayerNorm(HIDDEN), nn.LeakyReLU(),
                    nn.Linear(HIDDEN, cross_attention_dim)))
        self._packed = {}

    # ------------------------------------------------------------------------------------------
    def _params(self):
        out = []
        for i in range(self.num_tokens):
            for name in (f"mapping_{i}", f"mapping_patch_{i}"):
                seq = getattr(self, name)
                for li in (0, 1, 3, 4, 6):
                    out += [seq[li].weight, seq[li].bias]
        return out

    def _weights(self, dtype, device):
        """Stacked, compute-dtype copies of the weights: rebuilt only when a parameter's version changes."""
        params = self._params()
        key = tuple((p.data_ptr(), p._version) for p in params)
        pk = self._packed.get(dtype)
        if pk is not None and pk["key"] == key:
            return pk
        for p in params:
            if not p.is_cuda:
                raise RuntimeError("photoverse_b200 needs its weights on the CUDA device (no CPU fallback)")

        def m(t):   # fp32 master view (a cast happens only if the module was .to(bf16)'d)
            return t.detach().float().contiguous()
        T, D, E = self.num_tokens, self.clip_embedding_dim, self.cross_attention_dim
        pk = {"key": key}
        with torch.no_grad():
            for branch, prefix in (("cls", "mapping_"), ("patch", "mapping_patch_")):
                w1 = torch.empty(T, HIDDEN, D, device=device, dtype=dtype)
                w2 = torch.empty(T, HIDDEN, HIDDEN, device=device, dtype=dtype)
                for i in range(T):
                    seq = getattr(self, f"{prefix}{i}")
                    ops.pack_weight(m(seq[0].weight), w1[i])
                    ops.pack_weight(m(seq[3].weight), w2[i])
                pk[f"{branch}_w1"], pk[f"{branch}_w2"] = w1, w2
                for tag, li in (("b1", 0), ("g1", 1), ("b2", 3), ("g2", 4)):
                    pk[f"{branch}_{tag}"] = torch.stack(
                        [m(getattr(self, f"{prefix}{i}")[li].bias) if tag[0] == "b"
                         else m(getattr(self, f"{prefix}{i}")[li].weight) for i in range(T)]).contiguous()
                pk[f"{branch}_be1"] = torch.stack([m(getattr(self, f"{prefix}{i}")[1].bias) for i in range(T)]).contiguous()
                pk[f"{branch}_be2"] = torch.stack([m(getattr(self, f"{prefix}{i}")[4].bias) for i in range(T)]).contiguous()
            # last layer of both branches concatenated along K: [T, E, 2*HIDDEN]
            w3 = torch.empty(T, E, 2 * HIDDEN, device=device, dtype=dtype)
            tmp = torch.empty(E, HIDDEN, device=device, dtype=dtype)
            for i in range(T):
                w3[i, :, :HIDDEN] = ops.pack_weight(m(getattr(self, f"mapping_{i}")[6].weight), tmp)
                w3[i, :, HIDDEN:] = ops.pack_weight(m(getattr(self, f"mapping_patch_{i}")[6].weight), tmp)
            pk["w3"] = w3
            pk["b3"] = torch.stack([m(getattr(self, f"mapping_{i}")[6].bias)
                                    + m(getattr(self, f"mapping_patch_{i}")[6].bias) for i in range(T)]).contiguous()
        self._packed[dtype] = pk
        return pk

    # ------------------------------------------------------------------------------------------
    def _mlp2(self, x, pk, branch, sel, out2d, save):
        """Two (Linear -> LayerNorm -> LeakyReLU) layers for the selected heads.
        x: [T, M, D] -> writes the second activation into ``out2d`` ([T*M, HIDDEN] view, may be row-strided).
        Returns (x, h1, mean1, rstd1, a1, h2, mean2, rstd2); inference (``save`` False) reuses one fp32 buffer for both
        layers and keeps no statistics."""
        T, M, _ = x.shape
        dev = x.device
        h1 = torch.empty(T, M, HIDDEN, device=dev, dtype=torch.float32)
        a1 = torch.empty(T, M, HIDDEN, device=dev, dtype=x.dtype)
        h2 = torch.empty_like(h1) if save else h1
        ops.linear(x, pk[f"{branch}_w1"][sel], pk[f"{branch}_b1"][sel], out=h1)
        _, m1, r1 = ops.ln_lrelu(h1.view(T * M, HIDDEN), pk[f"{branch}_g1"][sel], pk[f"{branch}_be1"][sel],
                                 a1.view(T * M, HIDDEN), rows_per_group=M, eps=LN_EPS, slope=LRELU_SLOPE, save_stats=save)
        ops.linear(a1, pk[f"{branch}_w2"][sel], pk[f"{branch}_b2"][sel], out=h2)
        _, m2, r2 = ops.ln_lrelu(h2.view(T * M, HIDDEN), pk[f"{branch}_g2"][sel], pk[f"{branch}_be2"][sel], out2d,
                                 rows_per_group=M, eps=LN_EPS, slope=LRELU_SLOPE, save_stats=save)
        return x, h1, m1, r1, a1, h2, m2, r2

    def forward(self, embs: List[torch.Tensor], token_index: Optional[Union[int, str]] = None):
        if token_index is not None and token_index != "full":     # adapters.py:32-37
            heads = [int(token_index)]
            embs_sel = [embs[heads[0]]]
        else:                                                       # adapters.py:39-44
            embs_sel = list(embs)
            heads = list(range(len(embs_sel)))
            if len(heads) > self.num_tokens:
                raise AttributeError(f"adapter has {self.num_tokens} token heads, got {len(heads)} embeddings")
        e0 = embs_sel[0]
        if not e0.is_cuda:
            raise RuntimeError("photoverse_b200 runs on CUDA only (no CPU fallback)")
        if e0.dtype not in (torch.bfloat16, torch.float16, torch.float32):
            raise TypeError(f"embeddings must be bfloat16, float16 or float32, got {e0.dtype}")
        train = torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                             or any(e.requires_grad for e in embs_sel))
        # under CUDA autocast float32 embeddings compute in the autocast dtype (DESIGN.md 4.9): converted once per call,
        # differentiably where they require grad (which keeps that visible to adapter_autograd's check)
        autocast = ops.autocast_dtype() is not None
        dtype = ops.compute_dtype(e0.dtype, train)
        embs_sel = [_cast(e, dtype, autocast, e.requires_grad) for e in embs_sel]
        if train:
            if dtype == torch.float16:
                raise NotImplementedError(_F16_TRAINING)
            from .autograd import adapter_autograd
            return adapter_autograd(self, embs_sel, heads)
        return self._forward_impl(embs_sel, heads)

    def _forward_impl(self, embs_sel, heads, save=False):
        """The adapter on embeddings already in the compute dtype.  ``save``: also return what the backward needs,
        (packed weights, head slice, per-branch activations and statistics of :meth:`_mlp2`, cat)."""
        dtype, dev = embs_sel[0].dtype, embs_sel[0].device
        B, tokens, D = embs_sel[0].shape
        P = tokens - 1
        T = len(heads)
        pk = self._weights(dtype, dev)
        sel = slice(heads[0], heads[0] + 1) if T == 1 else slice(0, T)
        # gather the CLS rows and the patch rows of the selected heads (one strided copy each: plumbing)
        stacked = torch.stack(embs_sel) if T > 1 else embs_sel[0].unsqueeze(0)
        cls = stacked[:, :, 0, :].contiguous()                      # [T, B, D]
        patches = stacked[:, :, 1:, :].reshape(T, B * P, D)         # [T, B*P, D] (copy)
        cat = torch.empty(T, B, 2 * HIDDEN, device=dev, dtype=dtype)
        # CLS branch -> cat[..., :HIDDEN]
        saved = {"cls": self._mlp2(cls, pk, "cls", sel, cat.view(T * B, 2 * HIDDEN)[:, :HIDDEN], save)}
        # patch branch -> mean over the P patches -> cat[..., HIDDEN:]
        a2 = torch.empty(T * B * P, HIDDEN, device=dev, dtype=dtype)
        saved["patch"] = self._mlp2(patches, pk, "patch", sel, a2, save)
        ops.group_mean(a2.view(T * B, P, HIDDEN), cat.view(T * B, 2 * HIDDEN)[:, HIDDEN:])
        # last Linear of both branches in one K=2048 GEMM, written straight into [B, T, E]
        out = torch.empty(B, T, self.cross_attention_dim, device=dev, dtype=dtype)
        ops.linear(cat, pk["w3"][sel], pk["b3"][sel], out=out.permute(1, 0, 2))
        return (out, (pk, sel, saved, cat)) if save else out
