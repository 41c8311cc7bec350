"""The training step's kernels one by one, against fp64 references computed from the same rounded inputs, at the shapes
where they go wrong: ragged last tiles, the tile-per-CTA steps, every text length path of the attention backward, the
routing conditions of the weight gradient, the 64-row blocks of the LayerNorm partials.

The whole-layer tests (test_gpu_backward.py, test_gpu_train.py) bound a relative Frobenius norm over a full gradient tensor,
which still passes when a few rows out of thousands are wrong.  The metrics here are per row (attention backward) or per
element (weight gradients, reductions), so a single wrong boundary row, key slot or partial block fails.

Every bound carries, next to it, the largest value observed on one B200 (1000 W power limit) over all of its cases.
"""
import ctypes
import math

import pytest
import torch

LOG2E = 1.0 / math.log(2.0)
U32 = 2.0 ** -24                       # unit roundoff of fp32


def _rms(x: torch.Tensor) -> float:
    return x.double().square().mean().sqrt().item()


# ------------------------------------------------------------------------------------------------------------
# §1  attention-core backward (pv_dual_attn_bwd + pv_kv_pack_bwd) called directly
# ------------------------------------------------------------------------------------------------------------
def _segment_stats(q, kv_text, kv_img, B, Lt, Li, H):
    """(m, l) of each segment in the kernels' log2 domain: p = 2^(s scale log2e - m) / l, fp64 -> fp32 [B,H,S,4]."""
    S, C = q.shape[1], q.shape[2]
    d = C // H
    c = d ** -0.5 * LOG2E
    Q = q.double().view(B, S, H, d).transpose(1, 2)
    out = []
    for kv, L in ((kv_text, Lt), (kv_img, Li)):
        K = kv.double().view(B, L, 2, H, d)[:, :, 0].transpose(1, 2)
        s = Q @ K.transpose(-1, -2) * c
        m = s.amax(-1)
        out += [m, torch.exp2(s - m[..., None]).sum(-1)]
    return torch.stack(out, -1).float().contiguous()


def _attn_bwd_ref(q, d_o, kv_text, kv_img, d_vnorm, B, Lt, Li, H, w_key):
    """fp64 autograd of O = sum_seg sum_{k in seg} w_k softmax_seg(Q K^T / sqrt d)_k V_k with the loss <O, dO>, plus the
    derivative of <||V_img||, d_vnorm> written out: d_vnorm v / ||v|| (0 where ||v|| = 0).  ``w_key`` [Lt + Li] is the
    segment weight of every key slot (w_text on the text keys, w_img on the image keys).
    Returns (dQ [B,S,C], dkv_text [B*Lt,2C], dkv_img [B*Li,2C]) in fp64."""
    S, C = q.shape[1], q.shape[2]
    d = C // H
    with torch.enable_grad():
        qq = q.detach().double().requires_grad_(True)
        kt = kv_text.detach().double().requires_grad_(True)
        ki = kv_img.detach().double().requires_grad_(True)
        Q = qq.view(B, S, H, d).transpose(1, 2)
        o = 0.0
        for kv, L, w in ((kt, Lt, w_key[:Lt]), (ki, Li, w_key[Lt:])):
            K = kv.view(B, L, 2, H, d)[:, :, 0].transpose(1, 2)
            V = kv.view(B, L, 2, H, d)[:, :, 1].transpose(1, 2)
            p = torch.softmax(Q @ K.transpose(-1, -2) * d ** -0.5, -1)
            o = o + (p * w.to(p)) @ V
        loss = (o * d_o.detach().double().view(B, S, H, d).transpose(1, 2)).sum()
        dq, dkt, dki = torch.autograd.grad(loss, (qq, kt, ki))
    if d_vnorm is not None:
        v = kv_img.double().view(B, Li, 2, H, d)[:, :, 1]                    # [B, Li, H, d]
        n = v.norm(dim=-1, keepdim=True)
        dn = d_vnorm.double().transpose(1, 2)[..., None]                      # [B, Li, H, 1]
        term = torch.where(n > 0, dn * v / torch.where(n > 0, n, torch.ones_like(n)), torch.zeros_like(v))
        dki = dki.clone()
        dki.view(B, Li, 2, H, d)[:, :, 1] += term
    return dq, dkt, dki


def _row_errors(got, ref, floor_frac, row_floor=None):
    """||got - ref|| / max(||ref||, floor) over the last dimension; floor = floor_frac * RMS row norm of ref, or the larger
    per-row ``row_floor`` where one is given."""
    rn = ref.norm(dim=-1)
    floor = torch.full_like(rn, max(floor_frac * rn.square().mean().sqrt().item(), 1e-30))
    if row_floor is not None:
        floor = torch.maximum(floor, row_floor.to(floor))
    return (got - ref).norm(dim=-1) / torch.maximum(rn, floor), rn


def one_key_dk_scale(q, d_o, kv_text, kv_img, B, Lt, Li, H, w_key):
    """[B, L, H]: for the key of a ONE-key segment, the size of the terms whose cancellation makes its dK zero; 0 elsewhere.
    There p = 1, so ds_q = w (dp_q - delta_q) = w (dp_q - dp_q) for every query: the kernels compute p only to rounding
    and are left with ds_q ~ u w |dp_q|, i.e. dK ~ u scale ||sum_q w |dp_q| |Q_q|||.  That row is judged against this
    magnitude; the segment's weight or delta going wrong leaves a ds of the size of dp itself and fails."""
    S, C = q.shape[1], q.shape[2]
    d = C // H
    out = torch.zeros(B, Lt + Li, H, dtype=torch.float64, device=q.device)
    Q = q.double().view(B, S, H, d)
    dO = d_o.double().view(B, S, H, d)
    for kv, L, k0 in ((kv_text, Lt, 0), (kv_img, Li, Lt)):
        if L != 1:
            continue
        V = kv.double().view(B, 1, 2, H, d)[:, 0, 1]                          # [B, H, d]
        dp = (dO * V[:, None]).sum(-1).abs()                                  # [B, S, H]
        out[:, k0] = (w_key[k0].item() * d ** -0.5) * (dp[..., None] * Q.abs()).sum(1).norm(dim=-1)
    return out


FLOOR = 0.05        # per-row floor: 5 % of the RMS row norm (rows far below it are judged against it, not against 0)


def check_attn_bwd(got, ref, B, S, C, H, Lt, Li, bounds, w_key, dk_floor=None):
    """Per (query row, head) for dQ and per (sample, key slot, head) for dK / dV.  The keys of a zero-weight segment get
    no attention gradient at all: where their reference is 0 (dK always, dV without a norm term) the output must be 0 to
    1e-6.  (A segment of ONE key also has dK = 0, but only by cancellation, p = 1: that row is judged against
    ``dk_floor`` [B, L, H], the size of the cancelling terms, see one_key_dk_scale.)
    Returns (max errors, failures)."""
    d = C // H
    L = Lt + Li
    dq, dkt, dki = (t.double() for t in got)
    rq, rkt, rki = (t.double() for t in ref)
    fails = []
    for name, t in (("dQ", dq), ("dkv_text", dkt), ("dkv_img", dki)):
        if not torch.isfinite(t).all():
            fails.append(f"{name}: NaN / Inf")
    gk = torch.cat([dkt.view(B, Lt, 2, H, d), dki.view(B, Li, 2, H, d)], 1)
    rk = torch.cat([rkt.view(B, Lt, 2, H, d), rki.view(B, Li, 2, H, d)], 1)
    parts = {"dQ": (dq.view(B, S, H, d), rq.view(B, S, H, d)), "dK": (gk[:, :, 0], rk[:, :, 0]), "dV": (gk[:, :, 1], rk[:, :, 1])}
    worst = {}
    for name, (g, r) in parts.items():
        e, rn = _row_errors(g, r, FLOOR, dk_floor if name == "dK" else None)
        zero = rn == 0
        if name != "dQ":
            zero = zero & (w_key == 0).to(zero.device)[None, :, None]
        else:
            zero = torch.zeros_like(zero)
        if zero.any():
            z = g[zero].abs().max().item()
            if not z <= 1e-6:
                fails.append(f"{name}: {z:.3e} where the reference is exactly 0")
        e = torch.where(zero, torch.zeros_like(e), e)
        e = torch.nan_to_num(e, nan=float("inf"))
        worst[name] = e.max().item()
        if not worst[name] <= bounds[name]:
            idx = [int(i) for i in torch.nonzero(e == e.max())[0]]
            where = "(b, s, h)" if name == "dQ" else "(b, key, h)"
            fails.append(f"{name}: row error {worst[name]:.3e} > {bounds[name]:.1e} at {where} = {tuple(idx)} (of {tuple(e.shape)})")
    return worst, fails


# implementation -> (dtype, options, per-row bounds of the plain and of the peaked cases).  The largest error observed on
# the B200 over all cases is in the comment; each bound is 2-3x that.  The bf16 kernels round p and dS to bf16 for the
# tensor cores, the SIMT kernel keeps them in fp32.  In fp32, the peaked rows are ill-conditioned: at a nearly one-hot
# row dp - delta of the dominant key cancels to a small fraction of dp, so fp32 rounding of delta is amplified.
ATTN_IMPLS = {
    # default options: tcgen05 for head_dim 40 / 80, mma.sync for 160.  observed: dQ 5.6e-3 dK 4.7e-3 dV 4.5e-3
    "tcgen05-or-mma": (torch.bfloat16, {}, {"plain": {"dQ": 1.5e-2, "dK": 1.2e-2, "dV": 1.2e-2},
                                            "peaked": {"dQ": 1.5e-2, "dK": 1.2e-2, "dV": 1.2e-2}}),   # 4.7e-3 4.4e-3 3.9e-3
    # mma.sync for every head_dim.  observed: as above (the same kernel on most shapes' largest errors)
    "mma": (torch.bfloat16, {"bwd_tc": 0}, {"plain": {"dQ": 1.5e-2, "dK": 1.2e-2, "dV": 1.2e-2},
                                            "peaked": {"dQ": 1.5e-2, "dK": 1.2e-2, "dV": 1.2e-2}}),
    # SIMT kernel on bf16 inputs.  observed: dQ 2.8e-3 dK 2.9e-3 dV 2.6e-3 (peaked 2.5e-3 2.3e-3 2.4e-3)
    "simt-bf16": (torch.bfloat16, {"bwd_mma": 0}, {"plain": {"dQ": 7e-3, "dK": 7e-3, "dV": 7e-3},
                                                   "peaked": {"dQ": 7e-3, "dK": 7e-3, "dV": 7e-3}}),
    # fp32.  observed: dQ 1.5e-5 dK 2.2e-6 dV 1.5e-6; peaked dQ 3.6e-3 dK 1.3e-3 dV 2.5e-5
    "simt-f32": (torch.float32, {}, {"plain": {"dQ": 4e-5, "dK": 6e-6, "dV": 4e-6},
                                     "peaked": {"dQ": 1e-2, "dK": 3e-3, "dV": 6e-5}}),
}


def flags_kind(flags):
    return "peaked" if "peaked" in flags else "plain"

# (id, B, S, C, Lt, Li, w_text, w_img, flags); H = 8.  S covers the 2 / 4 / 8 tiles per CTA of the tcgen05 kernel
# (S < 512 / < 2048 / >= 2048), the 1 / 2 / 4 of mma.sync and ragged last tiles; Lt = 77 is the compile-time segment path.
ATTN_CASES = [
    ("s1_c320", 1, 1, 320, 77, 5, 1.0, 1.0, "vn"),
    ("s64_c640_lt1_li16", 3, 64, 640, 1, 16, 1.0, 1.0, ""),
    ("s127_c320_lt20_textonly", 3, 127, 320, 20, 1, 2.0, 0.0, ""),
    ("s128_c1280", 1, 128, 1280, 77, 5, 1.0, 1.0, "vn"),
    ("s129_c320_lt80_li16", 1, 129, 320, 80, 16, 1.0, 1.0, "vn"),
    ("s511_c640_lt76_imgonly", 3, 511, 640, 76, 5, 0.0, 2.0, "vn"),
    ("s512_c320_lt78_li16", 1, 512, 320, 78, 16, 1.3, 0.6, ""),
    ("s513_c640_li16_general", 3, 513, 640, 77, 16, 1.3, 0.6, "vn"),
    ("s513_c320_lt76_li1", 1, 513, 320, 76, 1, 1.0, 1.0, "vn"),
    ("s2047_c320_li1", 1, 2047, 320, 77, 1, 1.0, 1.0, "vn"),
    ("s2048_c640_lt20_textonly", 1, 2048, 640, 20, 5, 2.0, 0.0, ""),
    ("s2049_c320_general", 3, 2049, 320, 77, 5, 1.3, 0.6, "vn"),
    ("s2049_c640_lt78_li16", 1, 2049, 640, 78, 16, 1.0, 1.0, ""),
    ("s4096_c320_b16", 16, 4096, 320, 77, 5, 1.0, 1.0, "vn"),
    ("s4096_c640_lt20_li16", 1, 4096, 640, 20, 16, 0.7, 1.4, "vn"),
    ("s256_c1280_lt80_li16", 3, 256, 1280, 80, 16, 1.0, 1.0, "vn"),
    ("s1_c1280_lt1_li2_imgonly", 1, 1, 1280, 1, 2, 0.0, 2.0, ""),
    ("peaked_s700_c320", 1, 700, 320, 77, 5, 1.0, 1.0, "vn,peaked"),
    ("peaked_s129_c640_textonly", 1, 129, 640, 77, 16, 2.0, 0.0, "peaked"),
    ("zero_vrow_s300_c640", 3, 300, 640, 77, 5, 1.0, 1.0, "vn,zero_vrow"),
]


def _attn_inputs(case, dtype, device):
    name, B, S, C, Lt, Li, wt, wi, flags = case
    H = 8
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    # peaked: logits ~ 16x larger, so most softmax rows are nearly one-hot
    q = (torch.randn(B, S, C, generator=g) * (4.0 if "peaked" in flags else 1.0)).to(device, dtype)
    d_o = torch.randn(B, S, C, generator=g).to(device, dtype)
    kv_text = torch.randn(B * Lt, 2 * C, generator=g) * (4.0 if "peaked" in flags else 1.0)
    kv_img = torch.randn(B * Li, 2 * C, generator=g)
    if dtype == torch.bfloat16:         # the tensor-core kernels read K / V in bf16: give them values they hold exactly
        kv_text, kv_img = kv_text.bfloat16().float(), kv_img.bfloat16().float()
    if "zero_vrow" in flags:
        kv_img[Li + 1, C:] = 0.0        # sample 1, image key 1: all-zero value row, ||V|| = 0 in every head
    kv_text, kv_img = kv_text.to(device), kv_img.to(device)
    v_ip_norm = kv_img.double().view(B, Li, 2, H, C // H)[:, :, 1].norm(dim=-1).transpose(1, 2).float().contiguous()
    d_vnorm = torch.randn(B, H, Li, generator=g).to(device) if "vn" in flags else None
    stats = _segment_stats(q, kv_text, kv_img, B, Lt, Li, H)
    w_key = torch.tensor([wt] * Lt + [wi] * Li, dtype=torch.float64)
    return q, d_o, kv_text, kv_img, v_ip_norm, d_vnorm, stats, w_key


def _run_attn_bwd(q, d_o, kv_text, kv_img, stats, v_ip_norm, d_vnorm, H, Lt, Li, wt, wi):
    """One call with the shared workspace poisoned (0xFF bytes = NaN): a partial that is never written, or a chunk count
    that differs between the backward kernel and the K / V reduction, surfaces as NaN."""
    from photoverse_b200 import _lib, ops
    B, S, C = q.shape
    nbytes = _lib.lib().pv_dual_attn_bwd_ws_bytes(B, S, C, H, Lt, Li)
    ops._workspace(nbytes, q.device).fill_(0xFF)
    return ops.dual_attn_bwd(d_o, q, kv_text, kv_img, stats, v_ip_norm, d_vnorm, H, Lt, Li, wt, wi)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ATTN_CASES, ids=lambda c: c[0])
def test_attention_backward_kernels_per_row(cuda_device, case):
    from photoverse_b200 import _lib
    name, B, S, C, Lt, Li, wt, wi, flags = case
    H = 8
    fails = []
    ref_cache = {}
    for impl, (dtype, opts, bounds) in ATTN_IMPLS.items():
        q, d_o, kv_text, kv_img, v_ip_norm, d_vnorm, stats, w_key = _attn_inputs(case, dtype, cuda_device)
        if dtype not in ref_cache:
            ref_cache[dtype] = _attn_bwd_ref(q, d_o, kv_text, kv_img, d_vnorm, B, Lt, Li, H, w_key)
        ref = ref_cache[dtype]
        for k, v in opts.items():
            _lib.set_option(k, v)
        try:
            got = _run_attn_bwd(q, d_o, kv_text, kv_img, stats, v_ip_norm, d_vnorm, H, Lt, Li, wt, wi)
            again = _run_attn_bwd(q, d_o, kv_text, kv_img, stats, v_ip_norm, d_vnorm, H, Lt, Li, wt, wi)
        finally:
            _lib.set_option("bwd_tc", 1)
            _lib.set_option("bwd_mma", 1)
        dk_floor = one_key_dk_scale(q, d_o, kv_text, kv_img, B, Lt, Li, H, w_key)
        worst, f = check_attn_bwd(got, ref, B, S, C, H, Lt, Li, bounds[flags_kind(flags)], w_key, dk_floor)
        print(f"[attn-bwd] {name} {impl}: " + " ".join(f"{k}={v:.3e}" for k, v in worst.items()))
        fails += [f"{impl}: {m}" for m in f]
        for n_, a, b in zip(("dQ", "dkv_text", "dkv_img"), got, again):
            if not torch.equal(a, b):
                fails.append(f"{impl}: {n_} differs between two identical calls")
    assert not fails, "\n".join(fails)


def test_attention_backward_checker_rejects_small_mistakes():
    """CPU: the per-row checker passes the reference rounded to bf16 and fails each of these mutations at the loosest
    bf16 bound: one key slot's dK zeroed, one query row scaled by 1.03, dK / dV of one head swapped, and the segment
    weights of keys 76 (last text key) and 77 (first image key) exchanged."""
    B, S, C, H, Lt, Li, wt, wi = 1, 64, 320, 8, 77, 5, 1.3, 0.6
    case = ("selftest", B, S, C, Lt, Li, wt, wi, "vn")
    q, d_o, kv_text, kv_img, v_ip_norm, d_vnorm, stats, w_key = _attn_inputs(case, torch.bfloat16, torch.device("cpu"))
    ref = _attn_bwd_ref(q, d_o, kv_text, kv_img, d_vnorm, B, Lt, Li, H, w_key)
    loosest = {k: max(b[2][kind][k] for b in ATTN_IMPLS.values() for kind in ("plain", "peaked") if b[0] == torch.bfloat16)
               for k in ("dQ", "dK", "dV")}
    rounded = tuple(t.bfloat16() for t in ref)
    worst, fails = check_attn_bwd(rounded, ref, B, S, C, H, Lt, Li, loosest, w_key)
    assert not fails, fails
    d = C // H

    def mutated(fn):
        g = [t.double().clone() for t in rounded]
        fn(g)
        return check_attn_bwd(tuple(g), ref, B, S, C, H, Lt, Li, loosest, w_key)[1]

    def zero_key(g):                     # dK of text key slot 40, all heads
        g[1][40, :C] = 0.0

    def scale_row(g):                    # query row 37, head 3
        g[0][0, 37, 3 * d:4 * d] *= 1.03

    def swap_head(g):                    # dK <-> dV of head 2 in every text key slot
        k = g[1][:, 2 * d:3 * d].clone()
        g[1][:, 2 * d:3 * d] = g[1][:, C + 2 * d:C + 3 * d]
        g[1][:, C + 2 * d:C + 3 * d] = k

    assert mutated(zero_key)
    assert mutated(scale_row)
    assert mutated(swap_head)
    w_swapped = w_key.clone()
    w_swapped[76], w_swapped[77] = w_key[77], w_key[76]
    wrong = _attn_bwd_ref(q, d_o, kv_text, kv_img, d_vnorm, B, Lt, Li, H, w_swapped)
    assert check_attn_bwd(tuple(t.bfloat16() for t in wrong), ref, B, S, C, H, Lt, Li, loosest, w_key)[1]


# ------------------------------------------------------------------------------------------------------------
# §2  the softmax statistics the forward kernels save for the backward
# ------------------------------------------------------------------------------------------------------------
STATS_CASES = [                        # (id, dtype, B, S, C, Lt, Li): which forward kernel
    ("attn6_d40", torch.bfloat16, 2, 300, 320, 77, 1),
    ("attn6_d80", torch.bfloat16, 2, 384, 640, 20, 16),
    ("attn4_d160", torch.bfloat16, 2, 256, 1280, 77, 16),
    ("attn3_s_le_128", torch.bfloat16, 3, 100, 640, 20, 1),
    ("attn3_d160", torch.bfloat16, 2, 128, 1280, 77, 16),
    ("f32", torch.float32, 2, 200, 320, 77, 16),
    ("f32_d80", torch.float32, 1, 130, 640, 20, 1),
]
# |m + log2 l - log2sumexp2(logits)| in log2 units.  Largest observed: see the comment on each entry.
STATS_TOL = {torch.bfloat16: 1.5e-2,      # observed 5.1e-3 (Q rounded to bf16 in the kernel from its fp32 accumulator)
             torch.float32: 4e-6}        # observed 1.6e-6


@pytest.mark.gpu
@pytest.mark.parametrize("case", STATS_CASES, ids=lambda c: c[0])
def test_forward_saves_segment_statistics(cuda_device, case):
    from photoverse_b200 import _lib, ops
    name, dtype, B, S, C, Lt, Li = case
    H, Dc = 8, 768
    d = C // H
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    dev = cuda_device
    text = torch.randn(B, Lt, Dc, generator=g).to(dev, dtype)
    img = torch.randn(B, Li, Dc, generator=g).to(dev, dtype)
    wkv_t = (torch.randn(2 * C, Dc, generator=g) / Dc ** 0.5).to(dev, dtype)
    wkv_i = (torch.randn(2 * C, Dc, generator=g) / Dc ** 0.5).to(dev, dtype)
    x = torch.randn(B, S, C, generator=g).to(dev, dtype)
    wq = (torch.randn(C, C, generator=g) / C ** 0.5).to(dev, dtype)
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(dev, dtype)
    bo = torch.randn(C, generator=g).to(dev)
    kv = ops.kv_pack(text, img, wkv_t, wkv_i, H)
    # the logits the kernels see: bf16 Q = round(X Wq^T) and bf16-rounded K; fp32 keeps both in fp32
    if dtype == torch.bfloat16:
        q_bf16 = (x.double() @ wq.double().t()).to(dtype)
        kt, ki = kv.kv_text.to(dtype), kv.kv_img.to(dtype)
    else:
        kt, ki = kv.kv_text, kv.kv_img
    runs = {}                            # run -> (stats, the Q its logits come from)
    _, st = ops.dual_attn_core(x, wq, kv, 1.0, 1.0, want_stats=True)
    runs["core"] = (st, q_bf16 if dtype == torch.bfloat16 else x)             # fp32: the core takes Q itself
    for fuse in (2, 0):
        _lib.set_option("fuse_out", fuse)
        try:
            _, _, st, q32 = ops.dual_attn(x, wq, kv, wo, bo, 1.0, 1.0, want_stats=True)
        finally:
            _lib.set_option("fuse_out", 1)
        runs[f"fuse_out={fuse}"] = (st, q_bf16 if dtype == torch.bfloat16 else q32)   # fp32: its own projection
    fails = []
    for run, (st, qr) in runs.items():
        qd = qr.double().view(B, S, H, d).transpose(1, 2)
        for seg, kk, L in ((0, kt, Lt), (1, ki, Li)):
            K = kk.double().view(B, L, 2, H, d)[:, :, 0].transpose(1, 2)
            s = (qd @ K.transpose(-1, -2)) * (d ** -0.5 * LOG2E)
            lse = torch.logsumexp(s / LOG2E, -1) * LOG2E
            m, l_ = st[..., 2 * seg].double(), st[..., 2 * seg + 1].double()
            got = m + torch.log2(l_)
            if not torch.isfinite(got).all():
                fails.append(f"{run} segment {seg}: non-finite statistics")
                continue
            err = (got - lse).abs().max().item()
            print(f"[stats] {name} {run} seg{seg}: {err:.3e}")
            if not err <= STATS_TOL[dtype]:
                fails.append(f"{run} segment {seg}: |m + log2 l - lse2| = {err:.3e} > {STATS_TOL[dtype]}")
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------------------------------------
# §3  weight-gradient and reduction kernels
# ------------------------------------------------------------------------------------------------------------
def _poison_workspace(nbytes, device):
    from photoverse_b200 import ops
    ops._workspace(int(nbytes), device).fill_(0xFF)


# c in |got - ref| <= c u (|alpha| |G|^T |X| + |beta dW0|), u = 2^-24.  Largest observed c: see the comment on each entry.
WGRAD_C = {"tensor": 100.0,     # observed 40.6 (tcgen05, fp32 accumulation over K' = Mp)
           "simt": 12.0}        # observed 4.7 (fp32), 2.8 (bf16)


def _wgrad_route(dtype, M, N, K):
    """pv_bwd.cu linear_bwd_weight: transposes + tcgen05 GEMM, or the SIMT split-M kernel."""
    return "tensor" if (dtype == torch.bfloat16 and M >= 512 and N >= 128 and K >= 128 and N % 8 == 0 and K % 4 == 0) else "simt"


# (M, N, K, extra row stride of G, extra row stride of X): both sides of every routing condition, ragged Mp padding
WGRAD_SHAPES = [
    (511, 128, 128, 0, 0), (512, 128, 128, 0, 0), (513, 136, 132, 0, 0), (4103, 128, 128, 0, 0),
    (4103, 127, 128, 0, 0), (4103, 128, 126, 0, 0), (4103, 120, 128, 0, 0), (4103, 128, 124, 0, 0), (65536, 128, 128, 0, 0),
    (80, 640, 768, 0, 0),           # dkv_img [B*Li, 2C] x img (B = 16, Li = 5)
    (1232, 320, 128, 320, 0),       # rank-128 LoRA dB of to_k: g = dkv_text[:, :C] (ldg = 2C), t [M, 128]
    (1232, 128, 768, 0, 0),         # rank-128 LoRA dA of to_k: u [M, 128] x text
    (65536, 128, 320, 0, 0),        # rank-128 LoRA dA of to_q: u [B*S, 128] x x
    (65536, 320, 128, 0, 0),        # rank-128 LoRA dB of to_q: dQ [B*S, C] x t
    (2, 768, 2048, 0, 0),           # adapter out layer [B, 768] x [B, 2048]
    (512, 1024, 1024, 0, 0),        # adapter patch layers [256 B, 1024] x [256 B, 1024]
    (768, 1024, 1024, 0, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("M,N,K,xg,xx", WGRAD_SHAPES)
def test_linear_bwd_weight_elementwise(cuda_device, dtype, M, N, K, xg, xx):
    from photoverse_b200 import _lib, ops
    g = torch.Generator().manual_seed(M * 31 + N * 7 + K)
    G = torch.randn(M, N + xg, generator=g).to(cuda_device, dtype)[:, :N]
    X = torch.randn(M, K + xx, generator=g).to(cuda_device, dtype)[:, :K]
    route = _wgrad_route(dtype, M, N, K)
    dt = _lib.PV_BF16 if dtype == torch.bfloat16 else _lib.PV_F32
    nbytes = _lib.lib().pv_linear_bwd_weight_ws_bytes(dt, M, N, K)
    Gd, Xd = G.double(), X.double()
    mag = Gd.abs().t() @ Xd.abs()
    exact = Gd.t() @ Xd
    fails = []
    for alpha, beta in ((1.0, 0.0), (0.37, 0.0), (-1.5, 0.6)):
        w0 = torch.randn(N, K, generator=g).to(cuda_device) * mag.mean().item()
        out = w0.clone()
        _poison_workspace(nbytes, cuda_device)
        ops.linear_bwd_weight(G, X, out=out, alpha=alpha, beta=beta)
        ref = alpha * exact + beta * w0.double()
        bound = abs(alpha) * mag + abs(beta) * w0.double().abs()
        if not torch.isfinite(out).all():
            fails.append(f"alpha={alpha} beta={beta}: NaN / Inf")
            continue
        c = ((out.double() - ref).abs() / (U32 * bound).clamp_min(1e-30)).max().item()
        print(f"[wgrad] {route} {dtype} M={M} N={N} K={K} alpha={alpha} beta={beta}: c={c:.2f}")
        if not c <= WGRAD_C[route]:
            fails.append(f"{route} alpha={alpha} beta={beta}: error = {c:.1f} u |G|^T|X| > {WGRAD_C[route]} u")
    assert not fails, "\n".join(fails)


COLSUM_C = 24.0        # c in |got - ref| <= c u sum_m |G|.  observed 8.6 (fp32), 3.6 (bf16)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("M,N", [(1, 300), (255, 1000), (256, 768), (257, 1025), (20480, 320)])
def test_col_sum_elementwise(cuda_device, dtype, M, N):
    from photoverse_b200 import _lib, ops
    g = torch.Generator().manual_seed(M + N)
    G = (torch.randn(M, N + 24, generator=g) + 0.5).to(cuda_device, dtype)[:, 8:8 + N]      # strided, offset view
    _poison_workspace(_lib.lib().pv_col_sum_ws_bytes(M, N), cuda_device)
    out = ops.col_sum(G)
    ref = G.double().sum(0)
    bound = U32 * G.double().abs().sum(0)
    assert torch.isfinite(out).all()
    c = ((out.double() - ref).abs() / bound).max().item()
    print(f"[col_sum] {dtype} M={M} N={N}: c={c:.2f}")
    assert c <= COLSUM_C, f"error = {c:.1f} u sum|G| > {COLSUM_C} u"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("R", [1, 31, 33, 1280])
@pytest.mark.parametrize("C", [1, 31, 33, 1280])
def test_transpose_exact_and_padding_contract(cuda_device, dtype, R, C):
    from photoverse_b200 import _lib, ops
    g = torch.Generator().manual_seed(R * 3 + C)
    x = torch.randn(R, C + 7, generator=g).to(cuda_device, dtype)[:, :C]                    # ldi = C + 7 > C
    assert torch.equal(ops.transpose(x), x.t())
    # the C ABI's padded form (linear_bwd_weight's Mp rows): columns [R, ldo) zero-filled, nothing written past ldo * C
    ldo = R + 13
    guard = 300
    buf = torch.full((ldo * C + guard,), float("nan"), device=cuda_device, dtype=dtype)
    sentinel = buf.clone()
    dt = _lib.PV_BF16 if dtype == torch.bfloat16 else _lib.PV_F32
    _lib.check(_lib.lib().pv_transpose_2d(dt, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(buf.data_ptr()), R, C,
                                          x.stride(0), ldo, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
               "pv_transpose_2d")
    out = buf[:ldo * C].view(C, ldo)
    assert torch.equal(out[:, :R], x.t())
    assert torch.equal(out[:, R:], torch.zeros(C, ldo - R, device=cuda_device, dtype=dtype))
    assert torch.equal(buf[ldo * C:].view(torch.int16 if dtype == torch.bfloat16 else torch.int32),
                       sentinel[ldo * C:].view(torch.int16 if dtype == torch.bfloat16 else torch.int32))


@pytest.mark.gpu
def test_transpose_rejects_out_with_padded_rows(cuda_device):
    """ops.transpose would zero-fill columns [R, stride) of a row-padded ``out``: memory outside the view."""
    from photoverse_b200 import ops
    x = torch.randn(5, 3, device=cuda_device)
    buf = torch.full((3, 8), 7.0, device=cuda_device)
    with pytest.raises(ValueError):
        ops.transpose(x, buf[:, :5])
    assert torch.equal(buf, torch.full((3, 8), 7.0, device=cuda_device))
    out = torch.empty(3, 5, device=cuda_device)
    assert torch.equal(ops.transpose(x, out), x.t())


def _ln_lrelu_case(groups, rpg, slope, dtype, device, seed):
    g = torch.Generator().manual_seed(seed)
    cols = 1024
    rows = groups * rpg
    x = (torch.randn(rows, cols, generator=g) * 2 + 0.3).to(device)
    gamma = (1 + 0.2 * torch.randn(groups, cols, generator=g)).to(device)
    beta = (0.3 * torch.randn(groups, cols, generator=g)).to(device)
    xd = x.double()
    mean64 = xd.mean(1)
    rstd64 = 1.0 / torch.sqrt(xd.var(1, unbiased=False) + 1e-5)
    mean, rstd = mean64.float(), rstd64.float()
    xhat = (xd - mean64[:, None]) * rstd64[:, None]
    y = (xhat.view(groups, rpg, cols) * gamma.double()[:, None] + beta.double()[:, None]).view(rows, cols)
    da = torch.randn(rows, cols, generator=g).to(device)
    da = torch.where(y.abs() < 1e-3, torch.zeros_like(da), da).to(dtype)                   # no element on the kink
    return x, gamma, beta, mean, rstd, da


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("slope", [0.01, 0.2])
@pytest.mark.parametrize("groups,rpg", [(1, 1), (3, 2), (5, 63), (1, 64), (3, 65), (5, 256), (1, 4096), (3, 4096)])
def test_ln_lrelu_bwd_elementwise(cuda_device, dtype, slope, groups, rpg):
    from photoverse_b200 import _lib, ops
    x, gamma, beta, mean, rstd, da = _ln_lrelu_case(groups, rpg, slope, dtype, cuda_device, groups * 1000 + rpg)
    cols = 1024
    rows = groups * rpg
    _poison_workspace(_lib.lib().pv_ln_lrelu_bwd_ws_bytes(groups, rpg, cols), cuda_device)
    dx, dgamma, dbeta = ops.ln_lrelu_bwd(da, x, mean, rstd, gamma, beta, groups, rpg, slope)
    # fp64 reference from the same inputs (x fp32, da in its dtype; mean / rstd are the exact statistics of x)
    with torch.enable_grad():
        xd = x.double().requires_grad_(True)
        gd = gamma.double().requires_grad_(True)
        bd = beta.double().requires_grad_(True)
        h = torch.nn.functional.layer_norm(xd, (cols,), eps=1e-5).view(groups, rpg, cols) * gd[:, None] + bd[:, None]
        a = torch.nn.functional.leaky_relu(h, slope)
        rdx, rdg, rdb = torch.autograd.grad((a * da.double().view(groups, rpg, cols)).sum(), (xd, gd, bd))
    # magnitudes of the terms each output sums (forward-error bounds)
    with torch.no_grad():
        # |xhat| plus what fp32 (x - mean) rstd can lose to rounding: rstd (|x| + |mean|) u -- near the mean that is all
        xhat = ((x.double() - mean.double()[:, None]) * rstd.double()[:, None]).abs()
        xmag = (xhat + rstd.double()[:, None] * (x.double().abs() + mean.double().abs()[:, None])).view(groups, rpg, cols)
        gy = (da.double().view(groups, rpg, cols) * torch.where(h.detach() > 0, 1.0, slope)).abs()
        dxh = gy * gamma.double()[:, None].abs()
        mdx = rstd.double().view(groups, rpg, 1) * (dxh + dxh.mean(-1, keepdim=True) + xmag * (dxh * xmag).mean(-1, keepdim=True))
        mdg, mdb = (gy * xmag).sum(1), gy.sum(1)
    u_out = 2.0 ** -8 if dtype == torch.bfloat16 else U32           # rounding of dx to its dtype (half an ulp)
    assert torch.isfinite(dx).all() and torch.isfinite(dgamma).all() and torch.isfinite(dbeta).all()
    cdx = ((dx.double() - rdx).abs().view(groups, rpg, cols) / (LN_C["dx"] * U32 * mdx + u_out * rdx.abs().view(groups, rpg, cols)).clamp_min(1e-30)).max().item()
    cdg = ((dgamma.double() - rdg).abs() / (U32 * mdg).clamp_min(1e-30)).max().item()
    cdb = ((dbeta.double() - rdb).abs() / (U32 * mdb).clamp_min(1e-30)).max().item()
    print(f"[ln_lrelu_bwd] {dtype} slope={slope} groups={groups} rpg={rpg}: dx={cdx:.3f} (of bound) dgamma c={cdg:.2f} dbeta c={cdb:.2f}")
    assert cdx <= 1.0, f"dx error {cdx:.2f} x the bound"
    assert cdg <= LN_C["dgamma"], f"dgamma error {cdg:.1f} u sum|gy xhat| > {LN_C['dgamma']} u"
    assert cdb <= LN_C["dbeta"], f"dbeta error {cdb:.1f} u sum|gy| > {LN_C['dbeta']} u"


# c of the forward-error bounds of ln_lrelu_bwd (units of u = 2^-24).  Largest observed: see the comment on each entry.
LN_C = {"dx": 64.0,           # dx is bounded by its own bf16 rounding (observed 0.995 of the whole bound) or, in fp32, 0.05
        "dgamma": 64.0,       # observed 24 (before the rounding of xhat was part of the bound)
        "dbeta": 6.0}         # observed 2.2


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("groups,P,cols", [(3, 1, 1000), (2, 256, 1024), (5, 256, 300), (1, 7, 257)])
def test_group_mean_bwd_exact(cuda_device, dtype, groups, P, cols):
    from photoverse_b200 import ops
    g = torch.Generator().manual_seed(groups * P + cols)
    big = torch.randn(groups, 2 * cols + 3, generator=g).to(cuda_device, dtype)
    dy = big[:, cols + 3:]                          # the column slice the adapter passes (row stride > cols)
    dx = ops.group_mean_bwd(dy, P)
    # IEEE division (the build uses no fast-math).  Divide by a tensor: torch rewrites x / scalar as x * (1 / scalar),
    # which is not correctly rounded for P = 7.
    want = (dy.float() / torch.full_like(dy, P, dtype=torch.float32)).to(dtype)
    assert dx.shape == (groups, P, cols)
    assert torch.equal(dx, want[:, None, :].expand(groups, P, cols))


def _ulp(t: torch.Tensor, dtype) -> torch.Tensor:
    """One ulp of ``dtype`` at the magnitude of the fp64 tensor ``t``."""
    mant = 7 if dtype == torch.bfloat16 else 23
    tiny = torch.finfo(dtype).tiny
    e = torch.floor(torch.log2(t.abs().clamp_min(tiny)))
    return torch.exp2(e - mant)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("n", [8, (1 << 20) + 8 * 37])
def test_dropout_bwd_acc_within_one_ulp(cuda_device, dtype, p, n):
    from photoverse_b200 import ops
    g = torch.Generator().manual_seed(n + int(p * 10))
    dst = torch.randn(n, generator=g).to(cuda_device, dtype)
    src = torch.randn(n, generator=g).to(cuda_device, dtype)
    mask = (torch.rand(n, generator=g) >= p).to(cuda_device) if p > 0 else torch.ones(n, dtype=torch.bool, device=cuda_device)
    before = dst.clone()
    ops.dropout_bwd_acc(dst, src, mask, p)
    alpha = float(torch.tensor(1.0 / (1.0 - p), dtype=torch.float32))
    ref = before.double() + alpha * src.double()
    kept = mask
    err = (dst.double() - ref).abs()
    assert torch.equal(dst[~kept], before[~kept])
    assert bool((err[kept] <= _ulp(ref[kept], dtype)).all()), f"max error {(err[kept] / _ulp(ref[kept], dtype)).max().item():.2f} ulp"


# ------------------------------------------------------------------------------------------------------------
# §4  the GEMM shapes only the LoRA training paths use: N < 64 into a row-padded buffer (_skinny_linear)
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32], ids=["bf16-out", "f32-out"])
@pytest.mark.parametrize("M,N,K", [(4103, 4, 320), (1232, 4, 768), (300, 12, 1280)])
def test_linear_skinny_output_into_padded_rows(cuda_device, out_dtype, M, N, K):
    """x A^T (+ bias) with a LoRA rank N < 64, written into columns [0, N) of a row-padded buffer, as _skinny_linear does.
    The output tile is stored in whole 16-byte units: columns from N up to the next 16-byte boundary come out zero (the
    zero K extension _skinny_linear(full=True) hands to the following GEMM), columns past it stay untouched."""
    from photoverse_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g).to(cuda_device, torch.bfloat16)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_device, torch.bfloat16)
    bias = torch.randn(N, generator=g).to(cuda_device)
    per16 = 128 // torch.finfo(out_dtype).bits                      # elements per 16-byte unit
    n16 = (N + per16 - 1) // per16 * per16
    npad = n16 + 8
    buf = torch.full((M, npad), 3.0, device=cuda_device, dtype=out_dtype)
    ops.linear(a, w, bias, out=buf[:, :N])
    ref = a.double() @ w.double().t() + bias.double()
    mag = a.double().abs() @ w.double().abs().t() + bias.double().abs()
    u_out = 2.0 ** -8 if out_dtype == torch.bfloat16 else 0.0
    err = (buf[:, :N].double() - ref).abs() / (SKINNY_C * U32 * mag + u_out * ref.abs())
    print(f"[skinny] {out_dtype} M={M} N={N} K={K}: {err.max().item():.3f} of the bound")
    assert err.max().item() <= 1.0
    assert torch.equal(buf[:, N:n16], torch.zeros(M, n16 - N, device=cuda_device, dtype=out_dtype))
    assert torch.equal(buf[:, n16:], torch.full((M, npad - n16), 3.0, device=cuda_device, dtype=out_dtype))


SKINNY_C = 12.0      # c in |got - ref| <= c u |a| |w|^T (+ half an ulp of a bf16 output).  observed 4.5 (fp32 output)
