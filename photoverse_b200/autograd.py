"""Training path: ``torch.autograd.Function`` wrappers whose forward AND backward run in the CUDA library.

Reference semantics (train.py:495-538): gradients reach
  * the two adapters (every Linear / LayerNorm parameter),
  * ``to_k_ip`` / ``to_v_ip`` of the 16 processors (train.py:366-370),
  * the LoRA factors on ``attn2.to_q / to_k / to_v`` (train.py:348-354; peft: ``y = W x + scaling * B(A(x))``), and on
    ``attn2.to_out.0`` when it is a LoRA target too (the usual diffusers target set; the reference trains q/k/v only),
and flow through ``hidden_states`` / ``encoder_hidden_states`` into the rest of the (frozen) UNet, the text encoder and
the adapters.  The base projections and the base ``to_out`` weight and bias are frozen in every reference configuration;
asking for their gradients raises.

PyTorch is used for tensor ownership and autograd bookkeeping only: every contraction, reduction and elementwise
derivative below is a C-ABI call (photoverse_b200/csrc/pv_bwd.cu + the tcgen05 GEMM).
"""
from typing import List

import torch

from . import ops
from .adapters import HIDDEN, LRELU_SLOPE
from .attention_processor import _pad8
from .lora import linear_parts


def _skinny_linear(a2d: torch.Tensor, w: torch.Tensor, full: bool = False) -> torch.Tensor:
    """a2d [M,K] @ w[N,K]^T with a small N (LoRA rank): output rows padded to 16 bytes for the TMA store, view [M,N].
    ``full``: return the zero-padded [M, pad8(N)] buffer (usable as the K operand of a following GEMM)."""
    M, N = a2d.shape[0], w.shape[0]
    alloc = torch.zeros if (full and N % 8) else torch.empty
    buf = alloc(M, _pad8(N), device=a2d.device, dtype=a2d.dtype)
    out = buf[:, :N]
    ops.linear(a2d, w, out=out)
    return buf if full else out


def _pad_rows8(w: torch.Tensor) -> torch.Tensor:
    """[r, in] -> [pad8(r), in], zero rows appended (weight layout only)."""
    r = w.shape[0]
    if r % 8 == 0:
        return w.contiguous()
    out = torch.zeros(_pad8(r), w.shape[1], device=w.device, dtype=w.dtype)
    out[:r] = w
    return out


class _ConvertFn(torch.autograd.Function):
    """A float32 activation entering the 16-bit path under autocast (and its gradient leaving it): both directions are
    pv_convert_fwd."""

    @staticmethod
    def forward(ctx, x, dtype):
        ctx.src_dtype = x.dtype
        return ops.convert(x, dtype)

    @staticmethod
    def backward(ctx, g):
        return (g if g.dtype == ctx.src_dtype else ops.convert(g, ctx.src_dtype)), None


def convert(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Differentiable :func:`ops.convert`."""
    return _ConvertFn.apply(x, dtype)


class _DualAttnFn(torch.autograd.Function):
    """inputs: x, text, img, to_k_ip.w, to_v_ip.w, (A, B) of to_q, to_k, to_v, to_out[0] (None when not injected), ctx
    object.  LoRA is merged into the packed weights and the Q projection runs inside the attention kernel."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, x, text, img, w_kip, w_vip, qA, qB, kA, kB, vA, vB, oA, oB, meta):
        proc, attn = meta["proc"], meta["attn"]
        pk = proc._weights(attn, x.dtype, x.device)
        kv = ops.kv_pack(text, img, pk.wkv_text, pk.wkv_img, attn.heads)
        y, o, stats, q = ops.dual_attn(x, pk.wq, kv, pk.wo, pk.bo, meta["w_text"], meta["w_img"], want_stats=True)
        # fp32 mode keeps Q; the bf16 kernel never writes it (q is None: recomputed in backward).  O, the input of
        # to_out, is kept only for the gradients of a LoRA on to_out.
        _save(ctx, meta, pk, kv, stats, q, o if oA is not None else None,
              (x, text, img, w_kip, w_vip, qA, qB, kA, kB, vA, vB, oA, oB))
        return y, kv.v_ip_norm.clone()

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dy, dvn):
        meta, pk = ctx.meta, ctx.pk
        Lt, Li, H = ctx.dims
        x, text, img, stats, kv_text, kv_img, v_ip_norm, q, o, *rest = ctx.saved_tensors
        lora, drop = rest[:8], rest[8:]     # drop: dropout(input) of to_q / to_k / to_v / to_out, then their keep-masks
        dtype = x.dtype
        B, S, C = x.shape
        Dc = text.shape[2]
        x2, text2, img2 = x.view(B * S, C), text.view(B * Lt, Dc), img.view(B * Li, Dc)
        tw = _transposed(pk)
        need = ctx.needs_input_grad
        grads = [None] * 8

        dy2 = dy.contiguous().view(B * S, C).to(dtype)
        d_o = ops.linear(dy2, tw["wo_t"]).view(B, S, C)                                  # dO = dY Wo
        if lora[6] is not None:
            # LoRA on to_out: its factors from (O or dropout(O), dY); with dropout, the branch's share of dO before the
            # attention backward reads it.  The fusion rule never drops to_out.
            grads[6:8] = _lora_grads(o if o is None else o.view(B * S, C), dy2, d_o.view(B * S, C), True, lora[6], lora[7], meta["scal"][3], need[11],
                                     need[12], (drop[3], drop[7], meta["drop"][3]) if drop else None)
        if q is None:
            q = ops.linear(x2, pk.wq).view(B, S, C)                                      # recompute Q = X Wq^T
        d_vn = dvn if (dvn is not None and meta["vnorm_grad"]) else None
        dq, dkv_text, dkv_img = ops.dual_attn_bwd(d_o, q, kv_text, kv_img, stats, v_ip_norm, d_vn, H, Lt, Li,
                                                  meta["w_text"], meta["w_img"])
        dq2 = dq.view(B * S, C)
        dx = ops.linear(dq2, tw["wq_t"]) if need[0] else None                            # dX = dQ Wq (base weights)
        dtext = ops.linear(dkv_text, tw["wkv_text_t"]) if need[1] else None
        dimg = ops.linear(dkv_img, tw["wkv_img_t"]).view(B, Li, Dc) if need[2] else None
        # to_k_ip / to_v_ip : [dK_img | dV_img]^T img in one weight-gradient call -> rows [0, C) / [C, 2C)
        dkip = dvip = None
        if need[3] or need[4]:
            dkv_w = ops.linear_bwd_weight(dkv_img, img2)                     # [2C, Dc]
            dkip = dkv_w[:C] if need[3] else None
            dvip = dkv_w[C:] if need[4] else None
        srcs = ((x2, dq2, dx, need[0]), (text2, dkv_text[:, :C], dtext, need[1]), (text2, dkv_text[:, C:], dtext, need[1]))
        for j, (inp, g, dinp, need_inp) in enumerate(srcs):
            if lora[2 * j] is None or (j > 0 and not drop and meta["w_text"] == 0.0):
                continue                                                     # text branch dropped: no gradient (see below)
            grads[2 * j:2 * j + 2] = _lora_grads(inp, g, dinp, need_inp, lora[2 * j], lora[2 * j + 1], meta["scal"][j],
                                                 need[5 + 2 * j], need[6 + 2 * j],
                                                 (drop[j], drop[4 + j], meta["drop"][j]) if drop else None)
        dx = None if dx is None else dx.view(B, S, C)
        dtext = None if dtext is None else dtext.view(B, Lt, Dc)
        # A branch the fusion rule dropped (attention_processor.py:413-418) is not part of the reference's graph: its
        # parameters get NO gradient there (``.grad`` stays None and AdamW skips them -- no weight decay, no stale-momentum
        # update), not a zero one.  to_v_ip still receives the ``to_v_ip_norm`` regulariser term (:397, train.py:512-513).
        if meta["w_img"] == 0.0:
            dkip = None
            if dvn is None or not meta["vnorm_grad"]:
                dvip = None
        if meta["w_text"] == 0.0:
            grads[2:6] = [None] * 4                   # LoRA factors of to_k / to_v (text branch)
        pgrads = [None if gr is None else gr.to(dt) for gr, dt in zip((dkip, dvip, *grads), ctx.pdt)]
        return (dx, dtext, dimg, *pgrads, None)


class _DualAttnDropoutFn(_DualAttnFn):
    """Training step with LoRA dropout p > 0 (the reference default, train.py:264-269): peft's
    ``W x + s B A dropout(x)`` cannot be merged into one weight, so the low-rank branch rides along as a K-extension of
    the projection GEMMs: ``Q = [x | dropout(x) A^T] [W | s B]^T`` (same for K_text / V_text and the out projection
    ``Y = [O | dropout(O) A_o^T] [Wo | s B_o]^T + bo``, each with its own mask).

    The keep-masks come from ``torch.native_dropout`` -- the kernel ``nn.Dropout`` dispatches to -- drawn in the
    reference's order (to_q, to_k, to_v, then to_out after the attention; attention_processor.py:297, 304-305, 423) on
    same-shaped tensors, so a seeded run consumes the CUDA Philox stream exactly like the reference.  Everything
    downstream of the masks is C-ABI calls.
    The backward is :class:`_DualAttnFn`'s, with the LoRA factors' gradients taken from dropout(x) and the low-rank
    branch's input gradient added through the keep-masks."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, x, text, img, w_kip, w_vip, qA, qB, kA, kB, vA, vB, oA, oB, meta):
        proc, attn = meta["proc"], meta["attn"]
        dtype, dev = x.dtype, x.device
        u = proc._weights(attn, dtype, dev, merged=False)
        B, S, C = x.shape
        Lt, Li, Dc = text.shape[1], img.shape[1], text.shape[2]
        rq, rk, rv, ro = u.ranks
        pq, pk_, pv, po = meta["drop"]
        x2, text2 = x.view(B * S, C), text.view(B * Lt, Dc)

        def drop(t, p, has):
            if not has:
                return None, None
            if p > 0.0:
                return torch.native_dropout(t, p, True)
            return t, None

        xd_q, m_q = drop(x2, pq, qA is not None)
        xd_k, m_k = drop(text2, pk_, kA is not None)
        xd_v, m_v = drop(text2, pv, vA is not None)

        # Q = [x | xd A^T] [Wq | s B]^T
        if rq:
            xa = torch.empty(B * S, C + rq, device=dev, dtype=dtype)
            xa[:, :C] = x2
            ops.linear(xd_q, _pad_rows8(qA.detach().to(dtype)), out=xa[:, C:])
            q = ops.linear(xa, u.wq_aug).view(B, S, C)
            del xa
        else:
            q = ops.linear(x2, u.wq).view(B, S, C)
        # K/V of the text branch with their low-rank columns, image branch zero-extended to the same width
        if rk or rv:
            ta = torch.empty(B, Lt, Dc + rk + rv, device=dev, dtype=dtype)
            ta[..., :Dc] = text
            ta2 = ta.view(B * Lt, Dc + rk + rv)
            if rk:
                ops.linear(xd_k, _pad_rows8(kA.detach().to(dtype)), out=ta2[:, Dc:Dc + rk])
            if rv:
                ops.linear(xd_v, _pad_rows8(vA.detach().to(dtype)), out=ta2[:, Dc + rk:])
            ia = torch.zeros(B, Li, Dc + rk + rv, device=dev, dtype=dtype)
            ia[..., :Dc] = img
        else:
            ta, ia = text, img
        kv = ops.kv_pack(ta, ia, u.wkv_text_aug, u.wkv_img_aug, attn.heads)
        o, stats = ops.dual_attn_core(q, u.eye, kv, meta["w_text"], meta["w_img"], want_stats=True)
        o2 = o.view(B * S, C)
        od, m_o = drop(o2, po, oA is not None)           # drawn after the q / k / v masks, where the reference calls to_out
        # Y = [O | od A_o^T] [Wo | s B_o]^T + bo
        if ro:
            oa = torch.empty(B * S, C + ro, device=dev, dtype=dtype)
            oa[:, :C] = o2
            if oA.shape[0] % 8:
                oa[:, C + oA.shape[0]:].zero_()      # rank padding: fp32 rows of a rank-4 product end on a 16-byte boundary
            ops.linear(od, _pad_rows8(oA.detach().to(dtype)), out=oa[:, C:])
            y = ops.linear(oa, u.wo_aug, u.bo).view(B, S, C)
            del oa
        else:
            y = ops.linear(o2, u.wo, u.bo).view(B, S, C)
        _save(ctx, meta, u, kv, stats, q, None, (x, text, img, w_kip, w_vip, qA, qB, kA, kB, vA, vB, oA, oB),
              (xd_q, xd_k, xd_v, od, m_q, m_k, m_v, m_o))
        return y, kv.v_ip_norm.clone()


def _lora_grads(inp, g, dinp, need_inp, A, Bm, s, need_a, need_b, drop=None):
    """(dA, dB) of one LoRA-wrapped projection ``y = W inp + s B A inp`` from its input ``inp`` and ``g`` = dL/dy:
    dB = s g^T (inp A^T), dA = s (g B)^T inp.  ``drop`` = (dropout(inp), keep-mask or None, p) on the LoRA-dropout path:
    the factors see dropout(inp), and the branch's input gradient keep / (1 - p) * s (g B) A is added to ``dinp``."""
    dtype = g.dtype
    if drop is None:
        if need_a and need_b:
            fused = ops.lora_bwd(inp, g, A, Bm, s)                           # both factors, one pass over x and dY (rank <= 16)
            if fused is not None:
                return fused
    else:
        inp = drop[0]                                                        # dropout(x): what the branch saw
    dA = dB = None
    a_c = A.detach().to(dtype).contiguous()                                  # [r, in]
    bt_c = ops.transpose(Bm.detach().to(dtype).contiguous())                 # [r, out]
    if need_b:
        t = _skinny_linear(inp, a_c)                                         # x A^T            [M, r]
        dB = ops.linear_bwd_weight(g, t, alpha=s)                            # dB [out, r]
    grad_inp = drop is not None and need_inp
    if need_a or grad_inp:
        ub = _skinny_linear(g, bt_c, full=grad_inp)                          # dY B             [M, r] (padded: pad8(r))
        r = a_c.shape[0]
        if need_a:
            dA = ops.linear_bwd_weight(ub[:, :r], inp, alpha=s)              # dA [r, in]
        if grad_inp:
            # d dropout(x) = s (dY B) A, then through the mask:  d x += keep / (1 - p) * that
            at8 = ops.transpose(_pad_rows8(a_c * s))                         # [in, pad8(r)]
            v = ops.linear(ub, at8)                                          # [M, in]
            mask, p = drop[1], drop[2]
            if mask is not None:
                ops.dropout_bwd_acc(dinp, v, mask, p)
            else:
                ops.dropout_bwd_acc(dinp, v, torch.ones_like(v, dtype=torch.bool), 0.0)
    return dA, dB


def _save(ctx, meta, pk, kv, stats, q, o, inputs, drop=()):
    """What :meth:`_DualAttnFn.backward` reads: the pack the forward ran with (a re-pack makes a new object, so later
    parameter updates do not reach this backward), the saved tensors and the parameter dtypes of the gradients."""
    x, text, img, w_kip, w_vip, *lora = inputs
    ctx.meta, ctx.pk = meta, pk
    ctx.dims = (text.shape[1], img.shape[1], kv.H)
    ctx.save_for_backward(x, text, img, stats, kv.kv_text, kv.kv_img, kv.v_ip_norm, q, o, *lora, *drop)
    ctx.pdt = [None if t is None else t.dtype for t in (w_kip, w_vip, *lora)]


def _transposed(pk):
    """Transposed copies of the packed forward weights (the weights of the input-gradient GEMMs), cached per operand on the
    pack: the processor drops an entry when it re-packs that operand (attention_processor._weights)."""
    tw = pk._t
    for name in ("wq", "wo", "wkv_text", "wkv_img"):
        if name + "_t" not in tw:
            tw[name + "_t"] = ops.transpose(getattr(pk, name))
    return tw


def dual_attn_autograd(proc, attn, x, text, img, w_text, w_img):
    """Differentiable dual-branch attention: returns (Y [B,S,C], ||V_img|| [B,H,Li] fp32)."""
    frozen = [attn.to_out[0].bias]
    parts = [linear_parts(m) for m in (attn.to_q, attn.to_k, attn.to_v, attn.to_out[0])]
    frozen += [p[0] for p in parts]
    if any(t is not None and t.requires_grad for t in frozen):
        raise NotImplementedError(
            "gradients for the base attn2 projections / to_out are not part of the PhotoVerse training set "
            "(train.py:348-370 trains to_k_ip, to_v_ip and LoRA factors only)")
    meta = {"proc": proc, "attn": attn, "w_text": float(w_text), "w_img": float(w_img),
            "scal": [p[3] for p in parts], "drop": [p[4] for p in parts], "vnorm_grad": True}
    lora_args = []
    for p in parts:
        lora_args += [p[1], p[2]]
    fn = _DualAttnDropoutFn if max(meta["drop"]) > 0.0 else _DualAttnFn
    y, vn = fn.apply(x, text, img, proc.to_k_ip[0].weight, proc.to_v_ip[0].weight, *lora_args, meta)
    return y, vn


# ------------------------------------------------------------------------------------------------------------
# adapters
# ------------------------------------------------------------------------------------------------------------
class _AdapterFn(torch.autograd.Function):
    """inputs: meta, then for every selected head i, for (mapping_i, mapping_patch_i), for layer in (0,1,3,4,6):
    weight, bias  (20 tensors per head).  Embeddings (frozen CLIP states) are passed through ``meta``."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, meta, *params):
        out, ctx.saved = meta["adapter"]._forward_impl(meta["embs"], meta["heads"], save=True)
        ctx.meta = meta
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        meta = ctx.meta
        pk, sel, saved, cat = ctx.saved
        ad = meta["adapter"]
        T, B = cat.shape[:2]
        P = saved["patch"][0].shape[1] // B
        dtype = cat.dtype
        E = ad.cross_attention_dim
        tw = _adapter_transposed(pk, dtype)
        dout_t = dout.to(dtype).permute(1, 0, 2).contiguous()                       # [T, B, E]
        dcat = ops.linear(dout_t, tw["w3_t"][sel])                                  # [T, B, 2*HIDDEN]
        g = {}                                                                      # (head slot, branch, layer, 'w'|'b') -> grad
        for t in range(T):
            dw3 = ops.linear_bwd_weight(dout_t[t], cat[t])                          # [E, 2*HIDDEN]
            db3 = ops.col_sum(dout_t[t])
            g[(t, "cls", 6, "w")], g[(t, "patch", 6, "w")] = dw3[:, :HIDDEN], dw3[:, HIDDEN:]
            g[(t, "cls", 6, "b")] = g[(t, "patch", 6, "b")] = db3
        dcat2 = dcat.view(T * B, 2 * HIDDEN)
        for branch in ("cls", "patch"):
            x, h1, m1, r1, a1, h2, m2, r2 = saved[branch]
            M = x.shape[1]
            if branch == "cls":
                da2 = dcat2[:, :HIDDEN].contiguous()                                # [T*B, HIDDEN]
            else:
                da2 = ops.group_mean_bwd(dcat2[:, HIDDEN:], P).view(T * M, HIDDEN)  # mean over patches, backwards
            dh2, dg2, dbe2 = ops.ln_lrelu_bwd(da2, h2.view(T * M, HIDDEN), m2, r2, pk[f"{branch}_g2"][sel].contiguous(),
                                              pk[f"{branch}_be2"][sel].contiguous(), T, M, slope=LRELU_SLOPE)
            da1 = ops.linear(dh2.view(T, M, HIDDEN), tw[f"{branch}_w2_t"][sel])     # [T, M, HIDDEN]
            dh1, dg1, dbe1 = ops.ln_lrelu_bwd(da1.view(T * M, HIDDEN), h1.view(T * M, HIDDEN), m1, r1,
                                              pk[f"{branch}_g1"][sel].contiguous(), pk[f"{branch}_be1"][sel].contiguous(), T, M,
                                              slope=LRELU_SLOPE)
            dh2v, dh1v = dh2.view(T, M, HIDDEN), dh1.view(T, M, HIDDEN)
            for t in range(T):
                g[(t, branch, 3, "w")] = ops.linear_bwd_weight(dh2v[t], a1[t])
                g[(t, branch, 3, "b")] = ops.col_sum(dh2v[t])
                g[(t, branch, 0, "w")] = ops.linear_bwd_weight(dh1v[t], x[t])
                g[(t, branch, 0, "b")] = ops.col_sum(dh1v[t])
                g[(t, branch, 4, "w")], g[(t, branch, 4, "b")] = dg2[t], dbe2[t]
                g[(t, branch, 1, "w")], g[(t, branch, 1, "b")] = dg1[t], dbe1[t]
        grads = []
        params = meta["params"]
        k = 0
        for t in range(T):
            for branch in ("cls", "patch"):
                for li in (0, 1, 3, 4, 6):
                    for wb in ("w", "b"):
                        p = params[k]
                        grads.append(g[(t, branch, li, wb)].to(p.dtype).reshape(p.shape) if ctx.needs_input_grad[1 + k] else None)
                        k += 1
        return (None, *grads)


def _adapter_transposed(pk, dtype):
    tw = pk.get("_t")
    if tw is None:
        T = pk["w3"].shape[0]
        tw = {}
        for name in ("w3", "cls_w2", "patch_w2"):
            w = pk[name]                                            # [T, N, K]
            wt = torch.empty(T, w.shape[2], w.shape[1], device=w.device, dtype=w.dtype)
            for t in range(T):
                ops.transpose(w[t], wt[t])
            tw[name + "_t"] = wt
        pk["_t"] = tw
    return tw


def adapter_autograd(adapter, embs_sel: List[torch.Tensor], heads: List[int]):
    if any(e.requires_grad for e in embs_sel):
        raise NotImplementedError("gradients w.r.t. the CLIP hidden states are not needed on the PhotoVerse path "
                                  "(the image encoder is frozen and its outputs detached, train.py:487-492)")
    params = []
    for i in heads:
        for name in (f"mapping_{i}", f"mapping_patch_{i}"):
            seq = getattr(adapter, name)
            for li in (0, 1, 3, 4, 6):
                params += [seq[li].weight, seq[li].bias]
    meta = {"adapter": adapter, "embs": embs_sel, "heads": heads, "params": params}
    return _AdapterFn.apply(meta, *params)
