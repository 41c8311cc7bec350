"""Torch-tensor front end of the C ABI: pointer / stride marshalling only, no arithmetic.

PyTorch owns every buffer (inputs, outputs, workspaces); the native library gets raw device pointers and the
current CUDA stream.  Anything that is not a CUDA tensor of a supported dtype raises -- there is no fallback.
"""
import ctypes
from typing import Optional

import torch

from . import _lib
from ._lib import PV_BF16, PV_F16, PV_F32, PV_KEYS_PAD, check


_CODES = {torch.bfloat16: PV_BF16, torch.float32: PV_F32, torch.float16: PV_F16}
# the 16-bit compute dtypes: tensor-core kernels, fused Q projection, K/V operand tiles, single-launch processor
HALF_DTYPES = (torch.bfloat16, torch.float16)


def _code(dtype: torch.dtype) -> int:
    code = _CODES.get(dtype)
    if code is None:
        raise _lib.PhotoverseB200Error(f"unsupported dtype {dtype}: photoverse_b200 computes in bfloat16, float16 "
                                       "(inference only) or float32")
    return code


def _dt(t: torch.Tensor) -> int:
    return _code(t.dtype)


def _ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.PhotoverseB200Error("photoverse_b200 ops need CUDA tensors (no CPU fallback)")
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    assert t.dtype == torch.float32 and t.is_contiguous()
    return t


def resolve_compute_dtype(tensor_dtype: torch.dtype, grad_mode: bool, autocast_dtype: Optional[torch.dtype]) -> torch.dtype:
    """The dtype the processor and the adapters compute in (DESIGN.md 4.9).  ``autocast_dtype``: the dtype of the
    enclosing CUDA autocast region, None outside one.  Only float32 activations change dtype under autocast, and float16
    only without a backward pass (there is no fp16 backward): float32 in grad mode under fp16 autocast stays float32."""
    if autocast_dtype not in HALF_DTYPES or tensor_dtype != torch.float32:
        return tensor_dtype
    if autocast_dtype == torch.float16 and grad_mode:
        return torch.float32
    return autocast_dtype


def autocast_dtype() -> Optional[torch.dtype]:
    """The dtype of the enclosing CUDA autocast region, None outside one."""
    return torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None


def compute_dtype(tensor_dtype: torch.dtype, grad_mode: bool) -> torch.dtype:
    """:func:`resolve_compute_dtype` under the current CUDA autocast state."""
    return resolve_compute_dtype(tensor_dtype, grad_mode, autocast_dtype())


def convert(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """``x`` converted to ``dtype`` by pv_convert_fwd: float32 -> bfloat16 / float16 (round to nearest even, bit-identical
    to ``x.to(dtype)``) or bfloat16 / float16 -> float32 (exact).  Returns a new contiguous tensor."""
    if not x.is_cuda:
        raise _lib.PhotoverseB200Error("convert: CUDA tensor required (there is no CPU path)")
    src = x.contiguous()
    out = torch.empty(src.shape, device=src.device, dtype=dtype)
    check(_lib.lib().pv_convert_fwd(_dt(src), _code(dtype), _ptr(src), _ptr(out), src.numel(), _stream()), "pv_convert_fwd")
    return out


def pack_weight(w: torch.Tensor, out: torch.Tensor, lora_A=None, lora_B=None, scaling: float = 0.0) -> torch.Tensor:
    """out[out_f, in_f] (bf16|f16|f32) = w + scaling * lora_B @ lora_A  (fp32 masters)."""
    out_f, in_f = w.shape
    assert out.shape == w.shape and out.is_contiguous() and w.is_contiguous() and w.dtype == torch.float32
    r = 0
    if lora_A is not None:
        r = lora_A.shape[0]
        assert lora_A.shape == (r, in_f) and lora_B.shape == (out_f, r)
        lora_A, lora_B = _f32(lora_A.contiguous()), _f32(lora_B.contiguous())
    check(_lib.lib().pv_pack_weight(_dt(out), _ptr(w), _ptr(lora_A), _ptr(lora_B), float(scaling), _ptr(out),
                                    out_f, in_f, r, _stream()), "pv_pack_weight")
    return out


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None,
           out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """out[..., N] = a[..., K] @ w[..., N, K]^T + bias.  a: [M,K] or [batch,M,K]; w: [N,K] or [batch,N,K];
    bias fp32 [N] or [batch,N].  Inner-most dims must be contiguous; ``out`` may be a strided view whose rows are 16-byte
    aligned.  Rows are stored in whole 16-byte units: when N elements are not a multiple of 16 bytes, the columns from N up
    to the next 16-byte boundary of each row are set to zero (the zero K extension autograd._skinny_linear relies on)."""
    batched = a.dim() == 3
    if not batched:
        a3 = a.unsqueeze(0)
    else:
        a3 = a
    batch, M, K = a3.shape
    w3 = w if w.dim() == 3 else w.unsqueeze(0)
    N = w3.shape[1]
    assert w3.shape[2] == K and a3.stride(2) == 1 and w3.stride(2) == 1
    assert a.dtype == w.dtype, (a.dtype, w.dtype)
    if out_dtype is None:
        out_dtype = a.dtype if out is None else out.dtype
    if out is None:
        out = torch.empty((batch, M, N) if batched else (M, N), device=a.device, dtype=out_dtype)
    o3 = out if out.dim() == 3 else out.unsqueeze(0)
    assert o3.shape == (batch, M, N) and o3.stride(2) == 1
    stride_w = w3.stride(0) if (w.dim() == 3 and w3.shape[0] > 1) else 0
    if w.dim() == 3 and w3.shape[0] not in (1, batch):
        raise ValueError("weight batch must be 1 or match the activation batch")
    stride_b = 0
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.stride(-1) == 1
        stride_b = bias.stride(0) if (bias.dim() == 2 and bias.shape[0] > 1) else 0
    check(_lib.lib().pv_linear_fwd(_dt(a), _code(out_dtype), _ptr(a3), _ptr(w3), _ptr(bias), _ptr(o3),
                                   M, N, K, batch, a3.stride(1), w3.stride(1), o3.stride(1),
                                   a3.stride(0) if batch > 1 else 0, stride_w, stride_b,
                                   o3.stride(0) if batch > 1 else 0, _stream()), "pv_linear_fwd")
    return out


def kv_tile_bytes(dtype: torch.dtype, C: int, H: int, Lt: int, Li: int) -> int:
    n = int(_lib.lib().pv_kv_tile_bytes(_code(dtype), C, H, Lt, Li))
    if n <= 0:
        raise _lib.PhotoverseB200Error(f"bad K/V tile query C={C} H={H}")
    return n


class PackedKV:
    """Device buffers produced by :func:`kv_pack` (owned by PyTorch)."""
    __slots__ = ("Kp", "Vp", "v_ip_norm", "kv_text", "kv_img", "B", "Lt", "Li", "C", "H", "dtype", "_keepalive", "vnorm_act")


def kv_pack(text: torch.Tensor, img: torch.Tensor, wkv_text: torch.Tensor, wkv_img: torch.Tensor, H: int,
            out: Optional["PackedKV"] = None) -> PackedKV:
    """text [B,Lt,Dc], img [B,Li,Dc], wkv_* [2C,Dc] (all the compute dtype) -> packed K/V tiles + ||V_img||.
    ``out``: refresh an existing PackedKV of the same geometry in place (stable addresses for CUDA graphs)."""
    B, Lt, Dc = text.shape
    Li = img.shape[1]
    C = wkv_text.shape[0] // 2
    assert text.is_contiguous() and img.is_contiguous() and wkv_text.is_contiguous() and wkv_img.is_contiguous()
    assert text.dtype == img.dtype == wkv_text.dtype == wkv_img.dtype
    dev = text.device
    if out is not None and (out.B, out.Lt, out.Li, out.C, out.H, out.dtype) == (B, Lt, Li, C, H, text.dtype):
        kv = out
    else:
        kv = PackedKV()
        kv.B, kv.Lt, kv.Li, kv.C, kv.H, kv.dtype = B, Lt, Li, C, H, text.dtype
        tile = kv_tile_bytes(text.dtype, C, H, Lt, Li)
        kv.Kp = torch.empty(B * H * tile, device=dev, dtype=torch.uint8)
        kv.Vp = torch.empty(B * H * tile, device=dev, dtype=torch.uint8)
        kv.kv_text = torch.empty(B * Lt, 2 * C, device=dev, dtype=torch.float32)
        kv.kv_img = torch.empty(B * Li, 2 * C, device=dev, dtype=torch.float32)
        kv.v_ip_norm = torch.empty(B, H, Li, device=dev, dtype=torch.float32)
    check(_lib.lib().pv_kv_pack_fwd(_dt(text), _ptr(text), _ptr(img), _ptr(wkv_text), _ptr(wkv_img),
                                    _ptr(kv.kv_text), _ptr(kv.kv_img), _ptr(kv.Kp), _ptr(kv.Vp), _ptr(kv.v_ip_norm),
                                    B, Lt, Li, Dc, C, H, _stream()), "pv_kv_pack_fwd")
    # the processor's `to_v_ip_norm` side output in the activation dtype, [B,H,Li,1] (refreshed in place)
    if getattr(kv, "vnorm_act", None) is None:
        kv.vnorm_act = kv.v_ip_norm.to(text.dtype).unsqueeze(-1)
    else:
        kv.vnorm_act.copy_(kv.v_ip_norm.unsqueeze(-1))
    return kv


_SYNC = {}


def _sync_words(B: int, S: int, device) -> torch.Tensor:
    """Zeroed uint32 row-block counters of the single-launch processor kernel (include/photoverse_b200.h: ws_sync).
    One grow-only buffer per (device, stream): the kernel leaves it zeroed, calls on one stream are ordered."""
    need = int(_lib.lib().pv_dual_attn_sync_words(B, S))
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    buf = _SYNC.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.zeros(max(need, 1 << 16), device=device, dtype=torch.int32)
        _SYNC[key] = buf
    return buf


def dual_attn(x: torch.Tensor, wq: torch.Tensor, kv: PackedKV, wo: torch.Tensor, bo: torch.Tensor,
              w_text: float = 1.0, w_img: float = 1.0, want_stats: bool = False):
    """Y = (w_t softmax(QK_t^T/sqrt d) V_t + w_i softmax(QK_i^T/sqrt d) V_i) Wo^T + bo with Q = x Wq^T.
    Returns (Y, O, stats|None, Q|None); O (pre-out-projection) and Q (fp32 mode only) are kept for backward."""
    B, S, C = x.shape
    sync = _sync_words(B, S, x.device) if x.dtype in HALF_DTYPES else None
    assert x.is_contiguous() and wq.is_contiguous() and wo.is_contiguous()
    assert x.dtype == wq.dtype == wo.dtype == kv.dtype and bo.dtype == torch.float32
    assert (kv.B, kv.C) == (B, C)
    y = torch.empty_like(x)
    o = torch.empty_like(x)
    q = torch.empty(B, S, C, device=x.device, dtype=torch.float32) if x.dtype == torch.float32 else None
    stats = torch.empty(B, kv.H, S, 4, device=x.device, dtype=torch.float32) if want_stats else None
    check(_lib.lib().pv_dual_attn_fwd(_dt(x), _ptr(x), _ptr(wq), _ptr(kv.Kp), _ptr(kv.Vp), _ptr(wo), _ptr(bo),
                                      _ptr(y), _ptr(q), _ptr(o), _ptr(stats), _ptr(sync), B, S, C, kv.H, kv.Lt, kv.Li,
                                      float(w_text), float(w_img), _stream()), "pv_dual_attn_fwd")
    return y, o, stats, q


def dual_attn_core(x_or_q: torch.Tensor, wq: Optional[torch.Tensor], kv: PackedKV, w_text: float = 1.0,
                   w_img: float = 1.0, want_stats: bool = False):
    """The attention kernel alone (no out projection).  bf16 / fp16: ``x_or_q`` = X and ``wq`` is applied inside the
    kernel; fp32: ``x_or_q`` = Q (already projected), ``wq`` ignored.  Returns (O [B,S,C], stats|None)."""
    B, S, C = x_or_q.shape
    assert x_or_q.is_contiguous() and x_or_q.dtype == kv.dtype and (kv.B, kv.C) == (B, C)
    if x_or_q.dtype in HALF_DTYPES:
        assert wq is not None and wq.is_contiguous() and wq.dtype == x_or_q.dtype and wq.shape == (C, C)
    o = torch.empty_like(x_or_q)
    stats = torch.empty(B, kv.H, S, 4, device=o.device, dtype=torch.float32) if want_stats else None
    check(_lib.lib().pv_dual_attn_core_fwd(_dt(x_or_q), _ptr(x_or_q), _ptr(wq), _ptr(kv.Kp), _ptr(kv.Vp), _ptr(o),
                                           _ptr(stats), B, S, C, kv.H, kv.Lt, kv.Li, float(w_text), float(w_img),
                                           _stream()), "pv_dual_attn_core_fwd")
    return o, stats


def ln_lrelu(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor,
             rows_per_group: int = 0, eps: float = 1e-5, slope: float = 0.01, save_stats: bool = False):
    """out = leaky_relu(layer_norm(x) * gamma + beta); x fp32 [rows, cols] (row-strided ok), out bf16|f16|fp32."""
    rows, cols = x.shape
    assert x.dtype == torch.float32 and x.stride(1) == 1 and out.stride(1) == 1 and out.shape == x.shape
    assert gamma.dtype == beta.dtype == torch.float32 and gamma.is_contiguous() and beta.is_contiguous()
    mean = rstd = None
    if save_stats:
        mean = torch.empty(rows, device=x.device, dtype=torch.float32)
        rstd = torch.empty(rows, device=x.device, dtype=torch.float32)
    check(_lib.lib().pv_ln_lrelu_fwd(_dt(out), _ptr(x), _ptr(gamma), _ptr(beta), _ptr(out), _ptr(mean), _ptr(rstd),
                                     rows, cols, x.stride(0), out.stride(0), rows_per_group, eps, slope, _stream()),
          "pv_ln_lrelu_fwd")
    return out, mean, rstd


def group_mean(x: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """x [groups, P, cols] contiguous -> out [groups, cols] (row-strided ok) = mean over P."""
    groups, P, cols = x.shape
    assert x.is_contiguous() and out.shape == (groups, cols) and out.stride(1) == 1
    check(_lib.lib().pv_group_mean_fwd(_dt(x), _dt(out), _ptr(x), _ptr(out), groups, P, cols, out.stride(0),
                                       _stream()), "pv_group_mean_fwd")
    return out


# ------------------------------------------------------------------------------------------------------------
# backward ops (training step)
# ------------------------------------------------------------------------------------------------------------
_WS = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only per-device scratch buffer (stream-ordered re-use on the current stream)."""
    key = (device.type, device.index)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), device=device, dtype=torch.uint8)
        _WS[key] = buf
    return buf


def transpose(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[c, r] = x[r, c] for a 2-D tensor with contiguous rows.  ``out`` must have dense rows (row stride R): the kernel
    zero-fills every column up to the row stride, which for a row-padded ``out`` lies outside the view."""
    R, C = x.shape
    assert x.stride(1) == 1
    if out is None:
        out = torch.empty(C, R, device=x.device, dtype=x.dtype)
    assert out.shape == (C, R) and out.stride(1) == 1
    if out.stride(0) != R:
        raise ValueError(f"transpose: out must have row stride {R} (got {out.stride(0)}); columns up to the row stride "
                         "would be zero-filled")
    check(_lib.lib().pv_transpose_2d(_dt(x), _ptr(x), _ptr(out), R, C, x.stride(0), out.stride(0), _stream()), "pv_transpose_2d")
    return out


def linear_bwd_weight(g: torch.Tensor, x: torch.Tensor, out: Optional[torch.Tensor] = None, alpha: float = 1.0,
                      beta: float = 0.0) -> torch.Tensor:
    """dW[N,K] (fp32) = alpha * g^T x + beta * out;  g [M,N], x [M,K] (row-strided ok, same dtype)."""
    M, N = g.shape
    K = x.shape[1]
    assert x.shape[0] == M and g.dtype == x.dtype and g.stride(1) == 1 and x.stride(1) == 1
    if out is None:
        assert beta == 0.0
        out = torch.empty(N, K, device=g.device, dtype=torch.float32)
    assert out.shape == (N, K) and out.is_contiguous() and out.dtype == torch.float32
    lib = _lib.lib()
    ws = _workspace(lib.pv_linear_bwd_weight_ws_bytes(_dt(g), M, N, K), g.device)
    check(lib.pv_linear_bwd_weight(_dt(g), _ptr(g), _ptr(x), _ptr(out), _ptr(ws), M, N, K, g.stride(0), x.stride(0),
                                   float(alpha), float(beta), _stream()), "pv_linear_bwd_weight")
    return out


def lora_bwd(x: torch.Tensor, g: torch.Tensor, lora_A: torch.Tensor, lora_B: torch.Tensor, scaling: float):
    """(dA [r,in], dB [out,r]) fp32 of y = W x + scaling * B (A x), from x [M,in] and g = dL/dy [M,out] (row-strided ok),
    in ONE pass (rank <= 16); returns None when the shape needs the tensor-core route."""
    M, in_f = x.shape
    out_f = g.shape[1]
    r = lora_A.shape[0]
    assert g.shape[0] == M and x.dtype == g.dtype and x.stride(1) == 1 and g.stride(1) == 1
    assert lora_A.shape == (r, in_f) and lora_B.shape == (out_f, r)
    lib = _lib.lib()
    nbytes = int(lib.pv_lora_bwd_ws_bytes(M, in_f, out_f, r))
    if nbytes < 0:
        return None
    a32, b32 = _f32(lora_A.detach().float().contiguous()), _f32(lora_B.detach().float().contiguous())
    out = torch.empty(r * in_f + out_f * r, device=x.device, dtype=torch.float32)
    ws = _workspace(nbytes, x.device)
    check(lib.pv_lora_bwd(_dt(x), _ptr(x), _ptr(g), _ptr(a32), _ptr(b32), float(scaling), _ptr(out), _ptr(ws), M, in_f, out_f, r,
                          x.stride(0), g.stride(0), _stream()), "pv_lora_bwd")
    return out[:r * in_f].view(r, in_f), out[r * in_f:].view(out_f, r)


def col_sum(g: torch.Tensor) -> torch.Tensor:
    M, N = g.shape
    assert g.stride(1) == 1
    out = torch.empty(N, device=g.device, dtype=torch.float32)
    lib = _lib.lib()
    ws = _workspace(lib.pv_col_sum_ws_bytes(M, N), g.device)
    check(lib.pv_col_sum(_dt(g), _ptr(g), _ptr(out), _ptr(ws), M, N, g.stride(0), _stream()), "pv_col_sum")
    return out


def ln_lrelu_bwd(da: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, gamma: torch.Tensor,
                 beta: torch.Tensor, groups: int, rows_per_group: int, slope: float = 0.01):
    """Backward of ln_lrelu: da [rows, cols] (compute dtype, dense), x fp32 [rows, cols] -> (dx, dgamma, dbeta)."""
    rows, cols = da.shape
    assert rows == groups * rows_per_group and da.is_contiguous() and x.is_contiguous() and x.dtype == torch.float32
    dx = torch.empty_like(da)
    dgamma = torch.empty(groups, cols, device=da.device, dtype=torch.float32)
    dbeta = torch.empty_like(dgamma)
    lib = _lib.lib()
    ws = _workspace(lib.pv_ln_lrelu_bwd_ws_bytes(groups, rows_per_group, cols), da.device)
    check(lib.pv_ln_lrelu_bwd(_dt(da), _ptr(da), _ptr(x), _ptr(mean), _ptr(rstd), _ptr(gamma), _ptr(beta), _ptr(dx),
                              _ptr(dgamma), _ptr(dbeta), _ptr(ws), groups, rows_per_group, cols, float(slope), _stream()),
          "pv_ln_lrelu_bwd")
    return dx, dgamma, dbeta


def group_mean_bwd(dy: torch.Tensor, P: int) -> torch.Tensor:
    """dy [groups, cols] (row-strided ok) -> dx [groups, P, cols] = dy / P."""
    groups, cols = dy.shape
    assert dy.stride(1) == 1
    dx = torch.empty(groups, P, cols, device=dy.device, dtype=dy.dtype)
    check(_lib.lib().pv_group_mean_bwd(_dt(dy), _ptr(dy), _ptr(dx), groups, P, cols, dy.stride(0), _stream()),
          "pv_group_mean_bwd")
    return dx


def dual_attn_bwd(d_o: torch.Tensor, q: torch.Tensor, kv_text: torch.Tensor, kv_img: torch.Tensor, stats: torch.Tensor,
                  v_ip_norm: torch.Tensor, d_vnorm: Optional[torch.Tensor], H: int, Lt: int, Li: int, w_text: float,
                  w_img: float):
    """(dQ [B,S,C], dkv_text [B*Lt,2C], dkv_img [B*Li,2C]) in the compute dtype."""
    B, S, C = d_o.shape
    assert d_o.is_contiguous() and q.is_contiguous() and q.dtype == d_o.dtype and stats.is_contiguous()
    dq = torch.empty_like(d_o)
    dkv_text = torch.empty(B * Lt, 2 * C, device=d_o.device, dtype=d_o.dtype)
    dkv_img = torch.empty(B * Li, 2 * C, device=d_o.device, dtype=d_o.dtype)
    lib = _lib.lib()
    ws = _workspace(lib.pv_dual_attn_bwd_ws_bytes(B, S, C, H, Lt, Li), d_o.device)
    check(lib.pv_dual_attn_bwd(_dt(d_o), _ptr(d_o), _ptr(q), _ptr(kv_text), _ptr(kv_img), _ptr(stats), _ptr(dq), _ptr(ws),
                               B, S, C, H, Lt, Li, float(w_text), float(w_img), _stream()), "pv_dual_attn_bwd")
    if d_vnorm is not None:
        d_vnorm = d_vnorm.to(torch.float32).contiguous()
    check(lib.pv_kv_pack_bwd(_dt(d_o), _ptr(ws), _ptr(kv_img), _ptr(v_ip_norm), _ptr(d_vnorm), _ptr(dkv_text), _ptr(dkv_img),
                             B, S, Lt, Li, C, H, _stream()), "pv_kv_pack_bwd")
    return dq, dkv_text, dkv_img


def dropout_bwd_acc(dst: torch.Tensor, src: torch.Tensor, keep_mask: torch.Tensor, p: float) -> torch.Tensor:
    """dst += keep_mask * src / (1 - p): the input-gradient term of peft's LoRA dropout (in place on ``dst``)."""
    assert dst.is_contiguous() and src.is_contiguous() and keep_mask.is_contiguous()
    assert dst.shape == src.shape == keep_mask.shape and dst.dtype == src.dtype and keep_mask.dtype == torch.bool
    check(_lib.lib().pv_dropout_bwd_acc(_dt(dst), _ptr(dst), _ptr(src), _ptr(keep_mask), 1.0 / (1.0 - float(p)),
                                        dst.numel(), _stream()), "pv_dropout_bwd_acc")
    return dst


_SA_WS = {}


def self_attn(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int) -> torch.Tensor:
    """softmax(Q K^T / sqrt(d)) V per (sample, head) -- the stock self-attention of the ``attn1`` layers (reference
    models/unet.py:20-24 -> diffusers AttnProcessor2_0).  q, k, v: bf16 ``[B, S, C]`` views with unit channel stride and
    one common row stride (e.g. the three slices of a fused ``[B, S, 3C]`` projection); returns bf16 ``[B, S, C]``.
    Inference only (nothing is saved for a backward pass)."""
    if not (q.is_cuda and q.dtype == torch.bfloat16 and k.dtype == v.dtype == q.dtype):
        raise _lib.PhotoverseB200Error("self_attn: CUDA bfloat16 tensors required (there is no CPU path)")
    B, S, C = q.shape
    ld = q.stride(1)
    for t in (q, k, v):
        if t.shape != q.shape or t.stride(2) != 1 or t.stride(1) != ld or (B > 1 and t.stride(0) != S * ld):
            raise _lib.PhotoverseB200Error("self_attn: q, k, v must be [B,S,C] views with the same row stride and batch stride S*ld")
    lib = _lib.lib()
    nbytes = int(lib.pv_self_attn_ws_bytes(B, S, C, heads))
    if nbytes < 0:
        raise _lib.PhotoverseB200Error(f"self_attn: unsupported shape B={B} S={S} C={C} heads={heads}")
    key = (q.device.index, torch.cuda.current_stream(q.device).cuda_stream)
    ws = _SA_WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, device=q.device, dtype=torch.uint8)
        _SA_WS[key] = ws
    out = torch.empty(B, S, C, device=q.device, dtype=q.dtype)
    _lib.check(lib.pv_self_attn_fwd(_ptr(q), _ptr(k), _ptr(v), ld, _ptr(out), _ptr(ws), B, S, C, heads, _stream()), "pv_self_attn_fwd")
    return out


# ------------------------------------------------------------------------------------------------------------
# epilogues of the UNet evaluation around the path (SURVEY 8 row f1; inference only)
# ------------------------------------------------------------------------------------------------------------
def _gn_geometry(x: torch.Tensor, what: str):
    if not (x.is_cuda and x.dtype == torch.bfloat16):
        raise _lib.PhotoverseB200Error(f"{what}: CUDA bfloat16 activations required (there is no CPU path)")
    if x.dim() == 4:
        B, C, H, W = x.shape
        if not x.is_contiguous(memory_format=torch.channels_last):
            raise _lib.PhotoverseB200Error(f"{what}: the activation must be channels_last-contiguous")
        return B, H * W, C
    B, HW, C = x.shape
    if not x.is_contiguous():
        raise _lib.PhotoverseB200Error(f"{what}: [B, HW, C] input must be contiguous")
    return B, HW, C


def group_norm_nhwc(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, eps: float, silu: bool,
                    add: Optional[torch.Tensor] = None, save_stats: bool = False):
    """[SiLU](GroupNorm(x + add) * gamma + beta) of a ``torch.channels_last`` bf16 activation ``[B, C, H, W]`` (also accepts
    the equivalent dense ``[B, HW, C]``); gamma / beta fp32 ``[C]``; ``add``: optional fp32 ``[B, C]`` broadcast over the
    pixels.  The result has the layout of ``x``.  ``save_stats``: also return the fp32 ``[B, groups, 2]`` (mean, rstd)."""
    B, HW, C = _gn_geometry(x, "group_norm_nhwc")
    assert gamma.dtype == beta.dtype == torch.float32 and gamma.is_contiguous() and beta.is_contiguous() and gamma.numel() == C
    if add is not None:
        assert add.dtype == torch.float32 and add.is_contiguous() and add.shape == (B, C) and add.is_cuda
    lib = _lib.lib()
    nbytes = int(lib.pv_group_norm_nhwc_ws_bytes(B, HW, C, groups))
    if nbytes < 0:
        raise _lib.PhotoverseB200Error(f"group_norm_nhwc: unsupported shape B={B} HW={HW} C={C} groups={groups}")
    ws = torch.empty(nbytes, device=x.device, dtype=torch.uint8)
    y = torch.empty_like(x)                     # preserve_format: channels_last stays channels_last
    stats = torch.empty(B, groups, 2, device=x.device, dtype=torch.float32) if save_stats else None
    check(lib.pv_group_norm_nhwc_fwd(PV_BF16, _ptr(x), _ptr(add), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(stats), _ptr(ws), B, HW, C,
                                     groups, float(eps), 1 if silu else 0, _stream()), "pv_group_norm_nhwc_fwd")
    return (y, stats) if save_stats else y


def group_norm_nhwc_bwd(x: torch.Tensor, dy: torch.Tensor, stats: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor,
                        groups: int, silu: bool, add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Input gradient of :func:`group_norm_nhwc` (frozen affine): ``dy`` in the layout of ``x``."""
    B, HW, C = _gn_geometry(x, "group_norm_nhwc_bwd")
    # same shape and the same (channels-last / dense) layout; strides of size-1 dimensions are free to differ
    if dy.shape != x.shape or _gn_geometry(dy, "group_norm_nhwc_bwd") != (B, HW, C):
        raise _lib.PhotoverseB200Error("group_norm_nhwc_bwd: dy must have the shape, dtype and memory layout of x")
    assert stats.dtype == torch.float32 and stats.is_contiguous() and stats.shape == (B, groups, 2)
    lib = _lib.lib()
    ws = torch.empty(int(lib.pv_group_norm_nhwc_ws_bytes(B, HW, C, groups)), device=x.device, dtype=torch.uint8)
    dx = torch.empty_like(x)
    check(lib.pv_group_norm_nhwc_bwd(PV_BF16, _ptr(x), _ptr(add), _ptr(dy), _ptr(stats), _ptr(gamma), _ptr(beta), _ptr(dx), _ptr(ws),
                                     B, HW, C, groups, 1 if silu else 0, _stream()), "pv_group_norm_nhwc_bwd")
    return dx


def add_bias_nhwc(a: torch.Tensor, b: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``a + b + bias[c]`` for two bf16 activations of one shape and memory layout whose FASTEST dimension is the channel
    (channels_last ``[B, C, H, W]`` or dense ``[..., C]``); bias fp32 ``[C]``."""
    if not (a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.shape == b.shape):
        raise _lib.PhotoverseB200Error("add_bias_nhwc: two CUDA bfloat16 tensors of one shape required (there is no CPU path)")
    if a.dim() == 4:
        if not (a.is_contiguous(memory_format=torch.channels_last) and b.is_contiguous(memory_format=torch.channels_last)):
            raise _lib.PhotoverseB200Error("add_bias_nhwc: 4-D operands must be channels_last-contiguous")
        C = a.shape[1]
    else:
        if not (a.is_contiguous() and b.is_contiguous()):
            raise _lib.PhotoverseB200Error("add_bias_nhwc: operands must be contiguous")
        C = a.shape[-1]
    assert bias.dtype == torch.float32 and bias.is_contiguous() and bias.numel() == C
    out = torch.empty_like(a)
    check(_lib.lib().pv_add_bias_nhwc_fwd(PV_BF16, _ptr(a), _ptr(b), _ptr(bias), _ptr(out), a.numel() // C, C, _stream()),
          "pv_add_bias_nhwc_fwd")
    return out


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float) -> torch.Tensor:
    """LayerNorm over the last dimension of a contiguous bf16 ``[..., C]`` tensor (C <= 1280); gamma / beta fp32 ``[C]``."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and x.is_contiguous()):
        raise _lib.PhotoverseB200Error("layer_norm: contiguous CUDA bfloat16 input required (there is no CPU path)")
    C = x.shape[-1]
    assert gamma.dtype == beta.dtype == torch.float32 and gamma.is_contiguous() and beta.is_contiguous() and gamma.numel() == C
    y = torch.empty_like(x)
    check(_lib.lib().pv_layer_norm_fwd(PV_BF16, _ptr(x), None, None, _ptr(gamma), _ptr(beta), _ptr(y), x.numel() // C, C, float(eps),
                                       _stream()), "pv_layer_norm_fwd")
    return y


def add_layer_norm(x: torch.Tensor, residual: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float):
    """``s = x + residual`` (bf16) and ``LayerNorm(s)`` in one pass; returns ``(s, y)``."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and x.is_contiguous() and residual.dtype == x.dtype
            and residual.is_contiguous() and residual.shape == x.shape):
        raise _lib.PhotoverseB200Error("add_layer_norm: two contiguous CUDA bfloat16 tensors of one shape required")
    C = x.shape[-1]
    assert gamma.dtype == beta.dtype == torch.float32 and gamma.is_contiguous() and beta.is_contiguous() and gamma.numel() == C
    s, y = torch.empty_like(x), torch.empty_like(x)
    check(_lib.lib().pv_layer_norm_fwd(PV_BF16, _ptr(x), _ptr(residual), _ptr(s), _ptr(gamma), _ptr(beta), _ptr(y), x.numel() // C, C,
                                       float(eps), _stream()), "pv_layer_norm_fwd")
    return s, y


def layer_norm_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, eps: float) -> torch.Tensor:
    """Input gradient of :func:`layer_norm` (frozen affine) from the contiguous bf16 ``x`` and ``dy``."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and x.is_contiguous() and dy.dtype == x.dtype and dy.is_contiguous()
            and dy.shape == x.shape):
        raise _lib.PhotoverseB200Error("layer_norm_bwd: contiguous CUDA bfloat16 x and dy of one shape required")
    C = x.shape[-1]
    assert gamma.dtype == torch.float32 and gamma.is_contiguous() and gamma.numel() == C
    dx = torch.empty_like(x)
    check(_lib.lib().pv_layer_norm_bwd(PV_BF16, _ptr(x), _ptr(dy), _ptr(gamma), _ptr(dx), x.numel() // C, C, float(eps), _stream()),
          "pv_layer_norm_bwd")
    return dx


def geglu(h: torch.Tensor) -> torch.Tensor:
    """``h[..., :N] * gelu(h[..., N:])`` (exact GELU) of a bf16 projection ``[..., 2N]`` with contiguous rows."""
    if not (h.is_cuda and h.dtype == torch.bfloat16 and h.is_contiguous()):
        raise _lib.PhotoverseB200Error("geglu: contiguous CUDA bfloat16 input required (there is no CPU path)")
    N = h.shape[-1] // 2
    M = h.numel() // (2 * N)
    y = torch.empty(*h.shape[:-1], N, device=h.device, dtype=h.dtype)
    check(_lib.lib().pv_geglu_fwd(PV_BF16, _ptr(h), _ptr(y), M, N, 2 * N, _stream()), "pv_geglu_fwd")
    return y


def pack_geglu_weight(w: torch.Tensor, b: Optional[torch.Tensor]):
    """The ``nn.Linear(K, 2N)`` weight ``[2N, K]`` and bias of a GEGLU projection in the row order :func:`linear_geglu` reads:
    per 80 output columns j, the 80 value rows ``[80 j, 80 j + 80)`` then the 80 gate rows ``N + [80 j, 80 j + 80)``.
    Returns (bf16 contiguous weight, fp32 bias or None).  N % 80 == 0."""
    two_n, K = w.shape
    N = two_n // 2
    if two_n % 2 or N % 80:
        raise ValueError(f"pack_geglu_weight: need 2N rows with N % 80 == 0 (got {two_n})")
    def regroup(t):
        return torch.stack([t[:N].reshape(N // 80, 80, *t.shape[1:]), t[N:].reshape(N // 80, 80, *t.shape[1:])], 1).reshape(t.shape)
    wp = regroup(w.detach()).to(torch.bfloat16).contiguous()
    bp = None if b is None else regroup(b.detach()).float().contiguous()
    return wp, bp


def linear_geglu(x: torch.Tensor, w_packed: torch.Tensor, b_packed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``h[..., :N] * gelu(h[..., N:])`` with ``h = x @ W.T + b`` in one launch (the projection is never written):
    ``x`` ``[..., K]`` contiguous bf16; ``w_packed`` / ``b_packed`` from :func:`pack_geglu_weight`.  Rounds like
    ``linear`` to a bf16 ``h`` followed by :func:`geglu`."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and x.is_contiguous()):
        raise _lib.PhotoverseB200Error("linear_geglu: contiguous CUDA bfloat16 input required (there is no CPU path)")
    if not (w_packed.dtype == torch.bfloat16 and w_packed.dim() == 2 and w_packed.is_contiguous()):
        raise _lib.PhotoverseB200Error("linear_geglu: contiguous bfloat16 [2N, K] packed weight required")
    two_n, K = w_packed.shape
    if x.shape[-1] != K:
        raise _lib.PhotoverseB200Error(f"linear_geglu: input has {x.shape[-1]} features, the weight {K}")
    if b_packed is not None and not (b_packed.dtype == torch.float32 and b_packed.is_contiguous() and b_packed.numel() == two_n):
        raise _lib.PhotoverseB200Error("linear_geglu: contiguous float32 [2N] packed bias required")
    N = two_n // 2
    M = x.numel() // K
    y = torch.empty(*x.shape[:-1], N, device=x.device, dtype=x.dtype)
    check(_lib.lib().pv_linear_geglu_fwd(PV_BF16, _ptr(x), _ptr(w_packed), _ptr(b_packed), _ptr(y), M, N, K, K, N, _stream()),
          "pv_linear_geglu_fwd")
    return y


def geglu_bwd(h: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """Gradient of :func:`geglu` with respect to the ``[..., 2N]`` projection ``h`` from ``dy`` ``[..., N]`` (both contiguous bf16)."""
    if not (h.is_cuda and h.dtype == torch.bfloat16 and h.is_contiguous() and dy.dtype == h.dtype and dy.is_contiguous()):
        raise _lib.PhotoverseB200Error("geglu_bwd: contiguous CUDA bfloat16 h and dy required (there is no CPU path)")
    N = h.shape[-1] // 2
    M = h.numel() // (2 * N)
    assert dy.shape == (*h.shape[:-1], N)
    dh = torch.empty_like(h)
    check(_lib.lib().pv_geglu_bwd(PV_BF16, _ptr(h), _ptr(dy), _ptr(dh), M, N, 2 * N, _stream()), "pv_geglu_bwd")
    return dh
