"""The generation path's forward kernels one by one, against fp64 references computed from the operands as the kernels
round them, at the shapes where they go wrong: every routing family of the cross-attention core, ragged row blocks of
the out projection, the key tiles and the lazy-rescaling threshold of the self-attention kernel, both GEMM kernels under
every A/B switch, the packing and adapter epilogues.

The whole-layer tests (test_gpu_kernels.py, test_gpu_self_attn.py, test_gpu_f16.py) bound a max-abs error over a whole
output tensor, which a kernel with a 1 % error in one segment's weight, a one-sided rounding bias or a bf16 rounding
inside an fp16 kernel still passes.  The metrics here are per (sample, query row, head) for attention outputs, per
element for GEMMs and elementwise kernels, and a least-squares slope per softmax segment: the output is fitted as
a_t R_text + a_i R_img against the fp64 segment outputs R, and (a_t, a_i) must equal the segment weights (w_t, w_i).

Every bound carries, next to it, the largest value observed on one B200 (1000 W power limit) over all of its cases, and
is 2-3x that value (tools/gpu_runs/fwd_kernels_check.sh prints the maxima).  The GPU tests of this file take about 10 s
there (189 tests; measured with the same script).
"""
import ctypes
import math

import pytest
import torch

from tests.test_gpu_train_kernels import FLOOR, LOG2E, U32, _row_errors

H = 8
DC = 768                               # width of the text / image tokens (CLIP)
U_OUT = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 0.0}   # half an ulp, relative
DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _code(dtype):
    from photoverse_b200 import _lib
    return {torch.float32: _lib.PV_F32, torch.bfloat16: _lib.PV_BF16, torch.float16: _lib.PV_F16}[dtype]


def _trunc_bf16(t: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 by truncation (the low 16 bits dropped), back in fp64."""
    i = t.float().contiguous().view(torch.int32) & -65536
    return i.view(torch.float32).double()


def _ulp(t: torch.Tensor, dtype) -> torch.Tensor:
    """One ulp of ``dtype`` at the magnitude of the fp64 tensor ``t`` (subnormals: the ulp of the smallest normal)."""
    mant = {torch.bfloat16: 7, torch.float16: 10, torch.float32: 23}[dtype]
    e = torch.floor(torch.log2(t.abs().clamp_min(torch.finfo(dtype).tiny)))
    return torch.exp2(e - mant)


def _out_round(ref: torch.Tensor, dtype) -> torch.Tensor:
    """Bound of the rounding of an output to ``dtype``: half an ulp relative, and half the subnormal spacing."""
    if dtype == torch.float32:
        return torch.zeros_like(ref)
    return U_OUT[dtype] * ref.abs() + 0.5 * _ulp(torch.zeros_like(ref), dtype)


def _all_sync_counters_zero():
    from photoverse_b200 import ops
    return all(int(buf.abs().max().item()) == 0 for buf in ops._SYNC.values())


# ------------------------------------------------------------------------------------------------------------
# checkers (shared by the GPU tests and the CPU self-test of §7)
# ------------------------------------------------------------------------------------------------------------
def seg_slopes(got, r_text, r_img):
    """(a_t, a_i) of the least-squares fit got ~ a_t r_text + a_i r_img over the whole tensor."""
    g, a, b = got.double().flatten(), r_text.double().flatten(), r_img.double().flatten()
    m = torch.tensor([[a.dot(a).item(), a.dot(b).item()], [a.dot(b).item(), b.dot(b).item()]], dtype=torch.float64)
    rhs = torch.tensor([g.dot(a).item(), g.dot(b).item()], dtype=torch.float64)
    return torch.linalg.solve(m, rhs).tolist()


def slope_dev(alphas, ws):
    """Largest |a - w| relative to w (to the largest weight where w = 0)."""
    wmax = max(abs(w) for w in ws)
    return max(abs(a - w) / (abs(w) if w != 0 else wmax) for a, w in zip(alphas, ws))


TILE = 128          # query rows per tile of every attention kernel


def _tile_dots(x, y, B, S):
    """[B, ceil(S / 128)]: <x, y> over each 128-row query tile of each sample (zero rows pad the ragged last tile)."""
    T = (S + TILE - 1) // TILE
    pad = T * TILE - S
    xx = torch.nn.functional.pad(x.double().reshape(B, S, -1), (0, 0, 0, pad)).reshape(B, T, -1)
    yy = torch.nn.functional.pad(y.double().reshape(B, S, -1), (0, 0, 0, pad)).reshape(B, T, -1)
    return (xx * yy).sum(-1)


def tile_seg_slopes(got, r_text, r_img, B, S):
    """(a_t, a_i) of the least-squares fit of seg_slopes in every 128-row query tile: [B, T] each.  An error confined to
    one tile (the ragged last one, one CTA's unit) is diluted by the whole-tensor fit, not by this one."""
    aa, ab, bb = _tile_dots(r_text, r_text, B, S), _tile_dots(r_text, r_img, B, S), _tile_dots(r_img, r_img, B, S)
    ga, gb = _tile_dots(got, r_text, B, S), _tile_dots(got, r_img, B, S)
    det = aa * bb - ab * ab
    return (ga * bb - gb * ab) / det, (gb * aa - ga * ab) / det


def tile_slope_dev(alphas, ws):
    """slope_dev over every tile: the largest value and the (b, tile) where it is."""
    wmax = max(abs(w) for w in ws)
    dev = torch.stack([(a - w).abs() / (abs(w) if w != 0 else wmax) for a, w in zip(alphas, ws)]).amax(0)
    dev = torch.nan_to_num(dev, nan=float("inf"))
    return dev.max().item(), tuple(int(i) for i in torch.nonzero(dev == dev.max())[0])


def check_rows(got, ref, B, S, d, bounds, what):
    """Per (sample, query row, head): max and RMS over rows of ||got - ref|| / max(||ref||, 5 % of the RMS row norm).
    Returns (worst, failures)."""
    fails = []
    g = got.double().reshape(B, S, -1, d)
    r = ref.double().reshape(B, S, -1, d)
    if not torch.isfinite(g).all():
        fails.append(f"{what}: NaN / Inf (an unwritten row or tile?)")
        g = torch.nan_to_num(g, nan=1e30, posinf=1e30, neginf=-1e30)
    e, _ = _row_errors(g, r, FLOOR)
    worst = {"row": e.max().item(), "rms": e.square().mean().sqrt().item()}
    if not worst["row"] <= bounds["row"]:
        idx = tuple(int(i) for i in torch.nonzero(e == e.max())[0])
        fails.append(f"{what}: row error {worst['row']:.3e} > {bounds['row']:.1e} at (b, s, h) = {idx}")
    if not worst["rms"] <= bounds["rms"]:
        fails.append(f"{what}: RMS row error {worst['rms']:.3e} > {bounds['rms']:.1e}")
    return worst, fails


def check_cross(got, r_text, r_img, wt, wi, B, S, d, bounds, what):
    """Rows against w_t R_text + w_i R_img, and the segment slopes against (w_t, w_i)."""
    worst, fails = check_rows(got, wt * r_text + wi * r_img, B, S, d, bounds, what)
    if torch.isfinite(got).all():
        worst["slope"] = slope_dev(seg_slopes(got, r_text, r_img), (wt, wi))
        if not worst["slope"] <= bounds["slope"]:
            fails.append(f"{what}: segment slope off by {worst['slope']:.3e} > {bounds['slope']:.1e} (w = {wt}, {wi})")
        worst["tile_slope"], at = tile_slope_dev(tile_seg_slopes(got, r_text, r_img, B, S), (wt, wi))
        if not worst["tile_slope"] <= bounds["tile_slope"]:
            fails.append(f"{what}: segment slope of the row tile (b, tile) = {at} off by {worst['tile_slope']:.3e} > "
                         f"{bounds['tile_slope']:.1e} (w = {wt}, {wi})")
    return worst, fails


def check_self(got, ref, B, S, d, bounds, what):
    worst, fails = check_rows(got, ref, B, S, d, bounds, what)
    if torch.isfinite(got).all():
        g, r = got.double().flatten(), ref.double().flatten()
        worst["slope"] = abs(g.dot(r).item() / r.dot(r).item() - 1.0)
        if not worst["slope"] <= bounds["slope"]:
            fails.append(f"{what}: slope off by {worst['slope']:.3e} > {bounds['slope']:.1e}")
        dev = torch.nan_to_num((_tile_dots(got, ref, B, S) / _tile_dots(ref, ref, B, S) - 1.0).abs(), nan=float("inf"))
        worst["tile_slope"] = dev.max().item()
        if not worst["tile_slope"] <= bounds["tile_slope"]:
            at = tuple(int(i) for i in torch.nonzero(dev == dev.max())[0])
            fails.append(f"{what}: slope of the row tile (b, tile) = {at} off by {worst['tile_slope']:.3e} > {bounds['tile_slope']:.1e}")
    return worst, fails


def _fmt(worst):
    return " ".join(f"{k}={v:.3e}" for k, v in worst.items())


# ------------------------------------------------------------------------------------------------------------
# §1  cross-attention core: pv_dual_attn_core_fwd called directly
# ------------------------------------------------------------------------------------------------------------
def cross_segments(q, kv_text, kv_img, B, Lt, Li):
    """fp64 R_text, R_img [B, S, C] (each segment's softmax(Q K^T / sqrt d) V with unit weight) and the segments' log2
    sum-exp2 of the kernels' log2-domain logits, [B, H, S] each, from the rounded operands."""
    S, C = q.shape[1], q.shape[2]
    d = C // H
    Q = q.double().view(B, S, H, d).transpose(1, 2)
    rs, lses = [], []
    for kv, L in ((kv_text, Lt), (kv_img, Li)):
        K = kv.double().view(B, L, 2, H, d)[:, :, 0].transpose(1, 2)
        V = kv.double().view(B, L, 2, H, d)[:, :, 1].transpose(1, 2)
        s = Q @ K.transpose(-1, -2) * d ** -0.5
        rs.append((torch.softmax(s, -1) @ V).transpose(1, 2).reshape(B, S, C))
        lses.append(torch.logsumexp(s, -1) * LOG2E)
    return rs[0], rs[1], lses


def cross_model(q, kv_text, kv_img, B, Lt, Li, wt, wi, p_dtype=None, o_dtype=None, trunc=False, w_scale=(1.0, 1.0)):
    """CPU model of the kernels' rounding: per segment e = exp(s - max) (the max term is exactly 1), P = e rounded to
    ``p_dtype`` (or truncated to bf16 with ``trunc``), l = sum of the UNROUNDED e, O = sum_seg w (P V) / l rounded to
    ``o_dtype``.  ``w_scale`` multiplies the segment weights (a mutation of §7)."""
    S, C = q.shape[1], q.shape[2]
    d = C // H
    Q = q.double().view(B, S, H, d).transpose(1, 2)
    o = 0.0
    for kv, L, w in ((kv_text, Lt, wt * w_scale[0]), (kv_img, Li, wi * w_scale[1])):
        K = kv.double().view(B, L, 2, H, d)[:, :, 0].transpose(1, 2)
        V = kv.double().view(B, L, 2, H, d)[:, :, 1].transpose(1, 2)
        s = Q @ K.transpose(-1, -2) * d ** -0.5
        e = torch.exp(s - s.amax(-1, keepdim=True))
        p = _trunc_bf16(e) if trunc else (e.to(p_dtype).double() if p_dtype is not None else e)
        o = o + w * (p @ V) / e.sum(-1, keepdim=True)
    o = o.transpose(1, 2).reshape(B, S, C)
    return o.to(o_dtype).double() if o_dtype is not None else o


def cross_inputs(name, B, S, C, Lt, Li, flags):
    """fp32 CPU tensors (x, wq, text, img, wkv_text, wkv_img): logits of rms ~1, or ~16 with ``peaked`` (nearly one-hot
    rows); ``zero_img``: sample B - 1, image token 1 is all zero, so its K and V rows are 0 and ||V|| = 0 in every head."""
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    x = torch.randn(B, S, C, generator=g)
    wq = torch.randn(C, C, generator=g) / C ** 0.5
    text = torch.randn(B, Lt, DC, generator=g)
    img = torch.randn(B, Li, DC, generator=g)
    wkv_t = torch.randn(2 * C, DC, generator=g) / DC ** 0.5
    wkv_i = torch.randn(2 * C, DC, generator=g) / DC ** 0.5
    if "peaked" in flags:
        wq *= 4.0
        wkv_t[:C] *= 4.0
        wkv_i[:C] *= 4.0
    if "zero_img" in flags:
        img[B - 1, zero_token(Li)] = 0.0
    return x, wq, text, img, wkv_t, wkv_i


def zero_token(Li):
    return min(1, Li - 1)


def cross_family(dtype, S, C):
    """Which kernel pv_dual_attn_core_fwd reaches (pv_api.cu attn_core_bf16, pv_attn6.cu dual_attn_pair_roles_supported)."""
    if dtype == torch.float32:
        return "simt-f32"
    if S <= 128:
        return "attn3"
    d = C // H
    return "attn6" if (d == 40 and C == 320) or d == 80 else "attn4"


# (id, B, S, C, Lt, Li, flags); H = 8, so C = 320 / 640 / 1280 is head_dim 40 / 80 / 160.  Lt = 77 is the compile-time
# segment path of the CTA-pair kernels, 76 / 78 / 80 / 1 the run-time key mask.
CROSS_CASES = [
    ("s1_c320_lt77_li1", 3, 1, 320, 77, 1, ""),                 # attn3
    ("s64_c640_lt76_li16", 1, 64, 640, 76, 16, ""),             # attn3
    ("s127_c1280_lt78_li2", 3, 127, 1280, 78, 2, ""),           # attn3, head_dim 160
    ("s128_c320_lt1_li15", 1, 128, 320, 1, 15, ""),             # attn3, last S of the single-tile family
    ("s129_c320_lt80_li16", 3, 129, 320, 80, 16, ""),           # attn6 d = 40, one row past a tile
    ("s255_c640_lt77_li1", 1, 255, 640, 77, 1, ""),             # attn6 d = 80
    ("s256_c1280_lt76_li16", 3, 256, 1280, 76, 16, ""),         # attn4
    ("s257_c640_lt1_li2", 1, 257, 640, 1, 2, ""),               # attn6 d = 80, a ragged third row tile
    ("s513_c1280_lt80_li15", 1, 513, 1280, 80, 15, ""),         # attn4, odd row tile count
    ("s513_c320_lt78_li2", 3, 513, 320, 78, 2, ""),             # attn6 d = 40
    ("s4096_c320_lt77_li16", 2, 4096, 320, 77, 16, ""),         # attn6 d = 40, the SD-1.5 64^2 layer
    ("s4096_c640_lt76_li1", 1, 4096, 640, 76, 1, ""),           # attn6 d = 80
    ("b40_s256_c640_lt77_li1", 40, 256, 640, 77, 1, ""),        # attn6: 160 units for 74 CTA pairs
    ("b5_s300_c1280_lt77_li2", 5, 300, 1280, 77, 2, ""),        # attn4, odd B
    ("s2049_c1280_lt77_li5", 1, 2049, 1280, 77, 5, ""),         # attn4, ragged
    ("peaked_s700_c320_li16", 1, 700, 320, 77, 16, "peaked"),   # attn6
    ("peaked_s300_c640_lt76_li2", 2, 300, 640, 76, 2, "peaked"),
    ("peaked_s100_c1280_li5", 3, 100, 1280, 77, 5, "peaked"),   # attn3
    ("peaked_s257_c1280_li15", 1, 257, 1280, 78, 15, "peaked"),  # attn4
    ("zero_img_s300_c640", 3, 300, 640, 77, 5, "zero_img"),
    ("zero_img_s64_c320", 2, 64, 320, 77, 2, "zero_img"),
    ("zero_img_s300_c1280", 2, 300, 1280, 80, 16, "zero_img"),
]
WEIGHTS = [(1.0, 1.0), (2.0, 0.0), (0.0, 2.0), (1.3, 0.6)]

# dtype -> bounds of the rows (max and RMS over rows of the per-row error), of the segment slopes over the whole output
# and of the segment slopes per 128-row query tile.  The largest value observed on the B200 over all cases and weights
# (here and in the O of §2) is in the comment; each bound is 2-3x that.  The largest slopes come from the three-row case
# s1_c320, where few elements average the rounding out.
CROSS_BOUNDS = {
    # observed: row 4.9e-3, rms 2.5e-3, slope 4.5e-4, tile_slope 1.5e-3
    torch.bfloat16: {"row": 1.2e-2, "rms": 6e-3, "slope": 1.2e-3, "tile_slope": 3.5e-3},
    # observed: row 6.4e-4, rms 3.0e-4, slope 8.2e-5, tile_slope 2.3e-4 -- the fp16 rounding model: P or the O drain
    # rounded to bf16 inside an fp16 kernel gives row ~2.2e-3, rms ~1.3e-3 (the §7 self-test)
    torch.float16: {"row": 1.5e-3, "rms": 7e-4, "slope": 2e-4, "tile_slope": 6e-4},
    # observed: row 2.8e-5, rms 2.1e-6, slope 7.2e-8, tile_slope 1.8e-7 (the peaked rows: fp32 logits of size ~50)
    torch.float32: {"row": 7e-5, "rms": 5e-6, "slope": 2e-7, "tile_slope": 5e-7},
}
# |m + log2 l - log2sumexp2(logits)| of the saved statistics, in log2 units, from the same rounded Q and K
# observed: bf16 3.2e-5, fp16 4.2e-5, fp32 6.3e-5 (all in the peaked rows, fp32 logits of size ~50)
STATS_BOUNDS = {torch.bfloat16: 8e-5, torch.float16: 1e-4, torch.float32: 1.5e-4}


def _cross_operands(case, dtype, dev):
    """Device operands, the packed K / V and the rounded Q / K / V the kernel computes with."""
    from photoverse_b200 import ops
    name, B, S, C, Lt, Li, flags = case
    x, wq, text, img, wkv_t, wkv_i = cross_inputs(name, B, S, C, Lt, Li, flags)
    kv = ops.kv_pack(*(t.to(dev, dtype).contiguous() for t in (text, img, wkv_t, wkv_i)), H)
    xd, wqd = x.to(dev, dtype), wq.to(dev, dtype)
    if dtype == torch.float32:
        q = (x.double() @ wq.double().t()).float().to(dev)     # the fp32 core takes Q itself
        return q, None, kv, q, kv.kv_text, kv.kv_img
    # Q = round(X Wq^T) from an fp32 accumulator.  Rounded from fp64 instead, a few hundred elements of a large Q land on
    # the other side of a rounding boundary (a 2^-8 step of a logit, up to 1e-2 in a peaked row): the fp32 accumulator
    # comes from the library's GEMM, which sums the K blocks in the order of the kernel's fused projection (the saved
    # statistics then agree to 3e-5 instead of 5e-3).  A fault common to that GEMM and the fused projection would cancel
    # here; §4 checks the GEMM against fp64.
    q = ops.linear(xd.view(-1, C), wqd, out_dtype=torch.float32).view(B, S, C).to(dtype)
    return xd, wqd, kv, q, kv.kv_text.to(dtype), kv.kv_img.to(dtype)


def _core_call(dtype, xq, wq, kv, B, S, C, Lt, Li, wt, wi):
    """pv_dual_attn_core_fwd with O and the statistics pre-filled with NaN."""
    from photoverse_b200 import _lib
    o = torch.full((B, S, C), float("nan"), device=xq.device, dtype=dtype)
    st = torch.full((B, H, S, 4), float("nan"), device=xq.device, dtype=torch.float32)
    _lib.check(_lib.lib().pv_dual_attn_core_fwd(_code(dtype), _vp(xq), _vp(wq), _vp(kv.Kp), _vp(kv.Vp), _vp(o), _vp(st),
                                                B, S, C, H, Lt, Li, float(wt), float(wi), _stream()), "pv_dual_attn_core_fwd")
    return o, st


def check_stats(st, lses, bound, what):
    fails = []
    if not torch.isfinite(st).all():
        return float("inf"), [f"{what}: non-finite statistics (an unwritten row?)"]
    err = 0.0
    for seg in (0, 1):
        got = st[..., 2 * seg].double() + torch.log2(st[..., 2 * seg + 1].double())
        err = max(err, (got - lses[seg]).abs().max().item())
    if not err <= bound:
        fails.append(f"{what}: |m + log2 l - lse2| = {err:.3e} > {bound:.1e}")
    return err, fails


@pytest.mark.gpu
@pytest.mark.parametrize("case", CROSS_CASES, ids=lambda c: c[0])
def test_cross_attention_core_per_row(cuda_device, case):
    name, B, S, C, Lt, Li, flags = case
    d = C // H
    fails = []
    for dname, dtype in DTYPES.items():
        xq, wq, kv, q, kt, ki = _cross_operands(case, dtype, cuda_device)
        r_text, r_img, lses = cross_segments(q, kt, ki, B, Lt, Li)
        fam = cross_family(dtype, S, C)
        for wt, wi in WEIGHTS:
            o, st = _core_call(dtype, xq, wq, kv, B, S, C, Lt, Li, wt, wi)
            what = f"{fam} {dname} w=({wt},{wi})"
            worst, f = check_cross(o, r_text, r_img, wt, wi, B, S, d, CROSS_BOUNDS[dtype], what)
            worst["stats"], f2 = check_stats(st, lses, STATS_BOUNDS[dtype], what)
            print(f"[fwd:cross:{dname}] {name} {what}: {_fmt(worst)}")
            fails += f + f2
        if "zero_img" in flags:
            z = kv.v_ip_norm[B - 1, :, zero_token(Li)]
            if not torch.equal(z, torch.zeros_like(z)):
                fails.append(f"{dname}: ||V|| of the all-zero image token is {z.abs().max().item():.3e}, not 0")
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------------------------------------
# §2  out projection: the second phase of the attention launch (pv_outproj.cuh) and the GEMM launch (pv_gemm3.cu)
# ------------------------------------------------------------------------------------------------------------
OUTPROJ_C = {torch.bfloat16: 9.0, torch.float16: 9.0,     # observed 3.5 (bf16), 3.5 (fp16), either launch form
             torch.float32: 12.0}                           # observed 4.6
# c in |Y - ref| <= u_out |ref| + c u (|O| |Wo|^T + |bo|), ref = O_kernel Wo^T + bo in fp64


def _fwd_call(dtype, xq, wq, kv, wo, bo, B, S, C, Lt, Li, wt, wi):
    """pv_dual_attn_fwd with Y, O and the statistics pre-filled with NaN; returns (Y, O, stats, launches)."""
    from photoverse_b200 import _lib, ops
    dev = xq.device
    y = torch.full((B, S, C), float("nan"), device=dev, dtype=dtype)
    o = torch.full((B, S, C), float("nan"), device=dev, dtype=dtype)
    st = torch.full((B, H, S, 4), float("nan"), device=dev, dtype=torch.float32)
    ws_q = torch.full((B, S, C), float("nan"), device=dev, dtype=torch.float32) if dtype == torch.float32 else None
    sync = ops._sync_words(B, S, dev) if dtype != torch.float32 else None
    n0 = _lib.launch_count()
    _lib.check(_lib.lib().pv_dual_attn_fwd(_code(dtype), _vp(xq), _vp(wq), _vp(kv.Kp), _vp(kv.Vp), _vp(wo), _vp(bo), _vp(y),
                                           _vp(ws_q), _vp(o), _vp(st), _vp(sync), B, S, C, H, Lt, Li, float(wt), float(wi),
                                           _stream()), "pv_dual_attn_fwd")
    return y, o, st, _lib.launch_count() - n0


# (B, S, C, Lt, Li): C = 320 / 640 reach the fused pv_attn6 instances, C = 1280 the fused pv_attn4 instance (fuse_out = 2);
# S % 256 != 0 leaves a ragged last row block of the out-projection phase; S = 100 has one launch policy (attn3 + GEMM).
OUTPROJ_CASES = [(2, 300, 320, 77, 5), (1, 4103, 320, 76, 16), (3, 700, 640, 77, 1), (2, 1000, 640, 80, 16),
                 (2, 300, 1280, 77, 5), (1, 1100, 1280, 78, 2), (5, 257, 640, 77, 2), (2, 100, 640, 77, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16"])
@pytest.mark.parametrize("B,S,C,Lt,Li", OUTPROJ_CASES, ids=[f"B{b}_S{s}_C{c}_Lt{lt}_Li{li}" for b, s, c, lt, li in OUTPROJ_CASES])
def test_out_projection_both_launch_forms(cuda_device, dname, B, S, C, Lt, Li):
    from photoverse_b200 import _lib
    dtype = DTYPES[dname]
    d = C // H
    case = (f"op_{S}_{C}", B, S, C, Lt, Li, "")
    xq, wq, kv, q, kt, ki = _cross_operands(case, dtype, cuda_device)
    g = torch.Generator().manual_seed(S + C)
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(cuda_device, dtype)
    bo = torch.randn(C, generator=g).to(cuda_device)
    r_text, r_img, lses = cross_segments(q, kt, ki, B, Lt, Li)
    fails, ys = [], {}
    for wt, wi in ((1.0, 1.0), (1.3, 0.6)):
        for fuse in (2, 0):
            _lib.set_option("fuse_out", fuse)
            try:
                y, o, st, n = _fwd_call(dtype, xq, wq, kv, wo, bo, B, S, C, Lt, Li, wt, wi)
            finally:
                _lib.set_option("fuse_out", 1)
            form = "one-launch" if fuse == 2 and S > 128 else "two-launch"
            what = f"{dname} fuse_out={fuse} ({form}) w=({wt},{wi})"
            want = 1 if form == "one-launch" else 2
            if n != want:
                fails.append(f"{what}: {n} launches, the {form} form is {want}")
            if not _all_sync_counters_zero():
                fails.append(f"{what}: row-block counters not zero after the call")
            worst, f = check_cross(o, r_text, r_img, wt, wi, B, S, d, CROSS_BOUNDS[dtype], what + " O")
            worst["stats"], f2 = check_stats(st, lses, STATS_BOUNDS[dtype], what)
            fails += f + f2
            ref = o.double().view(-1, C) @ wo.double().t() + bo.double()
            mag = o.double().abs().view(-1, C) @ wo.double().abs().t() + bo.double().abs()
            yd = y.double().view(-1, C)
            if not torch.isfinite(yd).all():
                fails.append(f"{what}: Y has NaN / Inf (an unwritten row block?)")
                continue
            c = ((yd - ref).abs() - _out_round(ref, dtype)).clamp_min(0.0).div(U32 * mag).max().item()
            worst["c"] = c
            print(f"[fwd:outproj:{dname}] B{B} S{S} C{C} Lt{Lt} Li{Li} {what}: {_fmt(worst)}")
            if not c <= OUTPROJ_C[dtype]:
                fails.append(f"{what}: Y error {c:.1f} u (|O||Wo|^T + |bo|) beyond the output rounding > {OUTPROJ_C[dtype]}")
            ys[(wt, wi, fuse)] = (y, o)
        y2, o2 = ys[(wt, wi, 2)]
        y0, o0 = ys[(wt, wi, 0)]
        print(f"[fwd:outproj-identical:{dname}] B{B} S{S} C{C} w=({wt},{wi}): Y {torch.equal(y2, y0)} O {torch.equal(o2, o0)}")
        # the one-launch phase and the GEMM launch sum the same K blocks in the same order: bit-identical on the B200
        if not (torch.equal(y2, y0) and torch.equal(o2, o0)):
            fails.append(f"w=({wt},{wi}): the one-launch and the two-launch forms differ (Y {torch.equal(y2, y0)}, "
                         f"O {torch.equal(o2, o0)})")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
def test_out_projection_f32(cuda_device):
    """The fp32 parity path: Q projection GEMM, SIMT attention core, out-projection GEMM (three launches)."""
    B, S, C, Lt, Li = 2, 300, 640, 77, 5
    dtype = torch.float32
    case = ("op_f32", B, S, C, Lt, Li, "")
    xq, _, kv, q, kt, ki = _cross_operands(case, dtype, cuda_device)
    x, wq = (t.to(cuda_device) for t in cross_inputs(*case)[:2])
    g = torch.Generator().manual_seed(11)
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(cuda_device)
    bo = torch.randn(C, generator=g).to(cuda_device)
    y, o, st, n = _fwd_call(dtype, x, wq, kv, wo, bo, B, S, C, Lt, Li, 1.3, 0.6)
    assert n == 3
    ref = o.double().view(-1, C) @ wo.double().t() + bo.double()
    mag = o.double().abs().view(-1, C) @ wo.double().abs().t() + bo.double().abs()
    c = ((y.double().view(-1, C) - ref).abs() / (U32 * mag)).max().item()
    # O from the kernel's own fp32 Q projection: judged against the fp64 attention of the exact Q within the fp32 bound
    r_text, r_img, _ = cross_segments(q, kt, ki, B, Lt, Li)
    worst, fails = check_cross(o, r_text, r_img, 1.3, 0.6, B, S, C // H, CROSS_BOUNDS[dtype], "f32 O")
    print(f"[fwd:outproj:f32] B{B} S{S} C{C}: {_fmt(worst)} c={c:.3e}")
    assert not fails, "\n".join(fails)
    assert c <= OUTPROJ_C[dtype], c


# ------------------------------------------------------------------------------------------------------------
# §3  self-attention: pv_self_attn_fwd called directly
# ------------------------------------------------------------------------------------------------------------
# input family -> bounds.  "flat": q / k / v ~ 0.5 N(0, 1), logits of rms ~0.25: no key dominates a row, and P truncated
# to bf16 (pv_sattn.cu) is unbiased once numerator and denominator share it.  "plain": 1.5 N(0, 1) as the whole-layer
# test, rows where the maximum key holds a good share: its P is exactly 1 while every other P loses up to 2^-8 to the
# truncation, so the output leans towards the maximum key by ~1e-3 relative (a slope above 1) even with the shared
# denominator.  A denominator from the unrounded P shows as a slope below 1 (~2.8e-3) in the flat rows; in the plain
# rows the two leanings partly cancel and such a kernel cannot be told from a correct one, so the flat family, run at
# every shape, is the one that guards the cancellation.  Observed over all shapes and sattn_poly values (plain: with the
# structured rows of test_self_attention_rescaling_threshold_clamp_and_equal_logits):
SELF_BOUNDS = {"flat": {"row": 1.1e-2, "rms": 6e-3, "slope": 2e-4, "tile_slope": 1.3e-3},   # 4.3e-3 2.5e-3 7.3e-5 5.1e-4
               "plain": {"row": 1.3e-2, "rms": 6e-3, "slope": 1.2e-3, "tile_slope": 2.4e-3}}  # 5.1e-3 2.4e-3 4.8e-4 9.0e-4
SELF_SCALE = {"flat": 0.5, "plain": 1.5}


def self_ref(q, k, v, B, S, C):
    d = C // H
    f = lambda t: t.double().reshape(B, S, H, d).transpose(1, 2)
    s = f(q) @ f(k).transpose(-1, -2) * d ** -0.5
    return (torch.softmax(s, -1) @ f(v)).transpose(1, 2).reshape(B, S, C)


def self_model(q, k, v, B, S, C, bad_denominator=False):
    """CPU model of pv_sattn.cu: P truncated to bf16, numerator and denominator both contracted from that P (the ones
    column of V), output rounded to bf16.  ``bad_denominator``: the denominator from the unrounded P instead (§7)."""
    d = C // H
    f = lambda t: t.double().reshape(B, S, H, d).transpose(1, 2)
    s = f(q) @ f(k).transpose(-1, -2) * d ** -0.5
    e = torch.exp(s - s.amax(-1, keepdim=True))
    p = _trunc_bf16(e)
    o = (p @ f(v)) / (e if bad_denominator else p).sum(-1, keepdim=True)
    return o.transpose(1, 2).reshape(B, S, C).bfloat16().double()


def _self_call(q, k, v, B, S, C):
    """pv_self_attn_fwd with the operand-image workspace poisoned (0xFF bytes: NaN) and ``out`` pre-filled with NaN."""
    from photoverse_b200 import _lib
    lib = _lib.lib()
    nbytes = int(lib.pv_self_attn_ws_bytes(B, S, C, H))
    ws = torch.full((nbytes,), 0xFF, device=q.device, dtype=torch.uint8)
    out = torch.full((B, S, C), float("nan"), device=q.device, dtype=torch.bfloat16)
    _lib.check(lib.pv_self_attn_fwd(_vp(q), _vp(k), _vp(v), q.stride(1), _vp(out), _vp(ws), B, S, C, H, _stream()),
               "pv_self_attn_fwd")
    return out


SELF_SHAPES = [(c, s) for c in (320, 640, 1280) for s in (1, 63, 64, 65, 128, 255, 256, 257, 4095, 4096)]


@pytest.mark.gpu
@pytest.mark.parametrize("C,S", SELF_SHAPES, ids=[f"C{c}_S{s}" for c, s in SELF_SHAPES])
def test_self_attention_per_row(cuda_device, C, S):
    """64-key tiles (S = 63 / 64 / 65 ...), query units of 2 x 128 rows (S = 255 / 256 / 257), every sattn_poly variant."""
    from photoverse_b200 import _lib
    B = 2 if S < 4000 else 1
    fails = []
    for kind, scale in SELF_SCALE.items():
        g = torch.Generator().manual_seed(S * 7 + C)
        qkv = (torch.randn(B, S, 3 * C, generator=g) * scale).to(cuda_device, torch.bfloat16)
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        ref = self_ref(q, k, v, B, S, C)
        outs = {}
        try:
            for pf in (0, 2, 4):
                _lib.set_option("sattn_poly", pf)
                out = _self_call(q, k, v, B, S, C)
                worst, f = check_self(out, ref, B, S, C // H, SELF_BOUNDS[kind], f"{kind} sattn_poly={pf}")
                print(f"[fwd:self:{kind}] C{C} S{S} sattn_poly={pf}: {_fmt(worst)}")
                fails += f
                outs[pf] = out
        finally:
            _lib.set_option("sattn_poly", 2)
        # the sattn_poly variants compute the exponentials differently (MUFU or the FMA-pipe polynomial): on the B200 they
        # were bit-identical only where S = 1 (one key, P = 1), so each is judged against the bounds, not against the others
        print(f"[fwd:self-identical] C{C} S{S} {kind}: poly0==poly2 {torch.equal(outs[0], outs[2])} "
              f"poly4==poly2 {torch.equal(outs[4], outs[2])}")
    assert not fails, "\n".join(fails)


def self_structured_inputs(C):
    """B = 1, S = 257 (five key tiles, the last one ragged) with the head_dim-0 component carrying the structure:
    key 64 (the first of key tile 1) has k0 = J, every other key k0 = 0, and the query rows are
      rows   0..63 : q = e0      -> the running maximum jumps by J log2(e) / sqrt(d) at the key-tile boundary: just
                                    under the lazy-rescaling threshold 8 in heads 0..3, just over it in heads 4..7
      rows  64..127: q = 0       -> all logits equal
      rows 128..159: q = 20 e0   -> key 64 is ~160 (log2) above every other key: their exponentials hit the 2^-126 clamp
      rows 160..191: q = -20 e0  -> key 64 is ~160 below the maximum of tile 0
      rows 192..256: random."""
    d = C // H
    J = {40: (35.0, 35.25), 80: (49.5, 49.75), 160: (70.0, 70.5)}[d]
    scale = LOG2E / math.sqrt(d)
    assert J[0] * scale < 8.0 < J[1] * scale
    S = 257
    g = torch.Generator().manual_seed(C)
    q = torch.randn(1, S, C, generator=g) * 1.5
    k = torch.randn(1, S, C, generator=g) * 1.5
    v = torch.randn(1, S, C, generator=g)
    for h in range(H):
        c0 = h * d
        q[0, :192, c0:c0 + d] = 0.0
        q[0, :64, c0] = 1.0
        q[0, 128:160, c0] = 20.0
        q[0, 160:192, c0] = -20.0
        k[0, :, c0] = 0.0
        k[0, 64, c0] = J[0] if h < 4 else J[1]
    return q, k, v


@pytest.mark.gpu
@pytest.mark.parametrize("C", [320, 640, 1280])
def test_self_attention_rescaling_threshold_clamp_and_equal_logits(cuda_device, C):
    from photoverse_b200 import _lib
    q, k, v = (t.to(cuda_device, torch.bfloat16) for t in self_structured_inputs(C))
    B, S = 1, q.shape[1]
    ref = self_ref(q, k, v, B, S, C)
    fails = []
    try:
        for pf in (0, 2, 4):
            _lib.set_option("sattn_poly", pf)
            out = _self_call(q, k, v, B, S, C)
            worst, f = check_self(out, ref, B, S, C // H, SELF_BOUNDS["plain"], f"sattn_poly={pf}")
            # the structured row groups on their own
            for lo, hi, what in ((0, 64, "threshold"), (64, 128, "equal"), (128, 192, "clamp")):
                w2, f2 = check_rows(out[:, lo:hi], ref[:, lo:hi], B, hi - lo, C // H, SELF_BOUNDS["plain"], f"sattn_poly={pf} {what} rows")
                worst[what] = w2["row"]
                fails += f2
            print(f"[fwd:self-struct] C{C} sattn_poly={pf}: {_fmt(worst)}")
            fails += f
    finally:
        _lib.set_option("sattn_poly", 2)
    assert not fails, "\n".join(fails)


# ------------------------------------------------------------------------------------------------------------
# §4  GEMMs: pv_linear_fwd (pv_gemm.cu single-CTA kernel, pv_gemm3.cu persistent CTA-pair kernel), linear_geglu
# ------------------------------------------------------------------------------------------------------------
# c in |got - ref| <= u_out |ref| + c u (|A| |W|^T + |bias|), u = 2^-24
GEMM_C = 18.0       # observed 7.5 (fp16 in, fp32 out, K = 1288), 5.4 (bf16); the kv_pack workspaces of §5: 6.2

SWITCHES = [("default", {}), ("gemm_persistent=0", {"gemm_persistent": 0}), ("force_bn=64", {"force_bn": 64}),
            ("force_bn=128", {"force_bn": 128}), ("force_bn=160", {"force_bn": 160}), ("force_bn=256", {"force_bn": 256}),
            ("gemm_two_cta=0", {"gemm_two_cta": 0}), ("epi_swizzle=0", {"epi_swizzle": 0}), ("pdl=0", {"pdl": 0})]
SWITCH_DEFAULTS = {"gemm_persistent": 1, "force_bn": 0, "gemm_two_cta": 1, "epi_swizzle": 1, "pdl": 1}

# (M, N, K): M on both sides of the 128-row tiles, N on and off the BN choices (64 / 128 / 160 / 256) and 72, K from one
# 8-wide block to 1288 (K % 64 != 0).  (4103, 160 | 640, 320) reach the persistent kernel (16-bit out, M >= 512,
# N % 160 == 0, K % 64 == 0).
GEMM_SHAPES = [(1, 64, 8), (127, 72, 72), (128, 128, 320), (129, 160, 1288), (255, 256, 8), (256, 200, 72),
               (257, 320, 320), (4103, 640, 320), (4103, 160, 320), (4103, 72, 1288), (4103, 256, 72), (129, 64, 1288),
               (1, 160, 320), (4103, 128, 8)]


def _gemm_route(M, N, K, out_dtype, opts):
    o = dict(SWITCH_DEFAULTS, **opts)
    if (o["gemm_persistent"] and not o["force_bn"] and out_dtype != torch.float32 and M >= 512 and N % 160 == 0
            and K % 64 == 0):
        return "gemm3-pair"
    return "gemm-1cta"


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16"])
@pytest.mark.parametrize("M,N,K", GEMM_SHAPES, ids=[f"M{m}_N{n}_K{k}" for m, n, k in GEMM_SHAPES])
def test_linear_elementwise_every_switch(cuda_device, dname, M, N, K):
    from photoverse_b200 import _lib, ops
    dtype = DTYPES[dname]
    g = torch.Generator().manual_seed(M * 31 + N * 7 + K)
    a = torch.randn(M, K, generator=g).to(cuda_device, dtype)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_device, dtype)
    bias = torch.randn(N, generator=g).to(cuda_device)
    ref = a.double() @ w.double().t() + bias.double()
    mag = a.double().abs() @ w.double().abs().t() + bias.double().abs()
    fails = []
    for out_dtype in (dtype, torch.float32):
        base = None
        same = []
        for label, opts in SWITCHES:
            for k_, v_ in opts.items():
                _lib.set_option(k_, v_)
            try:
                out = torch.full((M, N), float("nan"), device=cuda_device, dtype=out_dtype)
                ops.linear(a, w, bias, out=out)
            finally:
                for k_, v_ in SWITCH_DEFAULTS.items():
                    _lib.set_option(k_, v_)
            route = _gemm_route(M, N, K, out_dtype, opts)
            what = f"{dname}->{str(out_dtype)[6:]} {label} ({route})"
            od = out.double()
            if not torch.isfinite(od).all():
                fails.append(f"{what}: NaN / Inf (an unwritten tile?)")
                continue
            c = ((od - ref).abs() - _out_round(ref, out_dtype)).clamp_min(0.0).div(U32 * mag).max().item()
            print(f"[fwd:gemm:{dname}] M{M} N{N} K{K} {what}: c={c:.2f}")
            if not c <= GEMM_C:
                fails.append(f"{what}: error {c:.1f} u |A||W|^T beyond the output rounding > {GEMM_C}")
            if base is None:
                base = out
            elif torch.equal(out, base):
                same.append(label)
            else:
                # every switch selects a kernel that sums the same K blocks in the same order: on the B200 each one was
                # bit-identical to the default at every shape, in both input and both output types
                fails.append(f"{what}: differs from the default options")
        print(f"[fwd:gemm-identical:{dname}] M{M} N{N} K{K} ->{str(out_dtype)[6:]}: bit-identical to default: {same}")
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", [(8, 8, 8), (512, 160, 64)], ids=["gemm-1cta", "gemm3-pair"])
def test_linear_f16_output_overflows_like_torch(cuda_device, M, N, K):
    """fp16 outputs at and past 65504: 65519 rounds to 65504, 65520 (the tie) and above to +-inf, as Tensor.to(float16)."""
    from photoverse_b200 import ops
    t = torch.tensor([0.0, 8.0, 15.0, 16.0, 31.0, 32.0, -65504.0, -16.0])
    a = torch.zeros(M, K)
    a[:, 0] = 65504.0
    a[:, 1] = t.repeat(M // 8 + 1)[:M]
    s = torch.tensor([[1.0, 1.0], [-1.0, -1.0], [1.0, 0.0], [0.5, 1.0], [1.0, -1.0], [-1.0, 0.0], [1.0, 0.5], [0.0, 1.0]])
    w = torch.zeros(N, K)
    w[:, :2] = s.repeat(N // 8 + 1, 1)[:N]
    want = (a @ w.t()).to(torch.float16)                     # small integers: the fp32 products and sums are exact
    assert torch.isinf(want).any() and (want.abs() == 65504).any()
    out = torch.full((M, N), float("nan"), device=cuda_device, dtype=torch.float16)
    ops.linear(a.to(cuda_device, torch.float16), w.to(cuda_device, torch.float16), None, out=out)
    assert torch.equal(out.cpu(), want)


GEGLU_C = GEMM_C    # c of the accumulation part of the bound below: the GEMM's.  Observed 0.77 of the whole bound


def geglu_model(x, wp, bp, N):
    """fp64 model of linear_geglu with its three rounding points: h = bf16(x W^T + b) (value and gate), gelu(h_gate)
    rounded to bf16, the product rounded to bf16.  Returns (model, exact fp64 h, |x| |W|^T + |b|), the latter two in the
    natural column order [value | gate]."""
    two_n = 2 * N
    j = torch.arange(N, device=wp.device)
    rows_a = (j // 80) * 160 + j % 80
    rows_g = rows_a + 80
    perm = torch.cat([rows_a, rows_g])
    w = wp[perm].double()
    b = bp[perm].double() if bp is not None else torch.zeros(two_n, dtype=torch.float64, device=wp.device)
    h = x.double() @ w.t() + b
    mag = x.double().abs() @ w.abs().t() + b.abs()
    hr = h.bfloat16().double()
    ge = (0.5 * hr[:, N:] * (1.0 + torch.erf(hr[:, N:] / math.sqrt(2.0)))).bfloat16().double()
    return (hr[:, :N] * ge).bfloat16().double(), h, mag


# (M, K, N): G = 2N / 160 column groups x V = ceil(M / 256) row units, shared out in ranges over 74 CTA pairs: the
# ranges cross from one column group into the next (the w_free wait of DESIGN 4.3) where G V is not a multiple of 74
GEGLU_SHAPES = [(8232, 320, 1280), (2000, 320, 1280), (4096, 640, 2560), (1000, 1280, 5120), (300, 320, 1280)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,K,N", GEGLU_SHAPES, ids=[f"M{m}_K{k}_N{n}" for m, k, n in GEGLU_SHAPES])
def test_linear_geglu_against_rounding_model(cuda_device, M, K, N):
    """Per element against the fp64 model.  A row of h whose fp32 accumulation lands on the other side of a bf16
    rounding boundary than the fp64 value moves by one bf16 ulp: the bound propagates one ulp of h_value / h_gate
    through the product plus the accumulation error, and the share of elements equal to the model is bounded below."""
    from photoverse_b200 import ops
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g).to(cuda_device, torch.bfloat16)
    w = (torch.randn(2 * N, K, generator=g) * 1.5 / K ** 0.5).to(cuda_device, torch.bfloat16)
    b = (0.3 * torch.randn(2 * N, generator=g)).to(cuda_device)
    wp, bp = ops.pack_geglu_weight(w, b)
    y = ops.linear_geglu(x, wp, bp)
    model, h, mag = geglu_model(x, wp, bp, N)
    assert torch.isfinite(y.float()).all()
    yd = y.double()
    ha, hg = h[:, :N], h[:, N:]
    gel = 0.5 * hg * (1.0 + torch.erf(hg / math.sqrt(2.0)))
    dgel = 0.5 * (1.0 + torch.erf(hg / math.sqrt(2.0))) + hg * torch.exp(-0.5 * hg * hg) / math.sqrt(2.0 * math.pi)
    da = _ulp(ha, torch.bfloat16) + GEGLU_C * U32 * mag[:, :N]
    dg = _ulp(hg, torch.bfloat16) + GEGLU_C * U32 * mag[:, N:]
    bound = gel.abs() * da + ha.abs() * (dgel.abs() * dg + _ulp(gel, torch.bfloat16)) + _ulp(model, torch.bfloat16) + da * dg
    frac = ((yd - model).abs() / bound).max().item()
    eq = (yd == model).double().mean().item()
    print(f"[fwd:geglu] M{M} K{K} N{N}: {frac:.3f} of the bound, {eq:.4f} equal to the model")
    assert frac <= 1.0
    assert eq >= 0.99                                # observed 0.9964: 0.36 % of the elements off the model


# ------------------------------------------------------------------------------------------------------------
# §5  packing and adapter epilogues
# ------------------------------------------------------------------------------------------------------------
# c in |W_eff - (W + s B A)| <= c u (|W| + s |B| |A|) of the fp32 sum of r products: observed 1.8 (r = 1), 2.7 (r = 4),
# 3.6 (r = 16).  The 16-bit outputs: within one ulp of the rounded fp64 value beyond that (observed exactly 1.00 ulp
# where the fp32 sum and the fp64 value round to neighbours)
def PACK_C(r):
    return 0.4 * r + 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("r", [0, 1, 4, 16])
def test_pack_weight_within_one_ulp(cuda_device, dname, r):
    from photoverse_b200 import ops
    dtype = DTYPES[dname]
    g = torch.Generator().manual_seed(r + 3)
    out_f, in_f = 640, 772
    w = (torch.randn(out_f, in_f, generator=g) * 0.05).to(cuda_device)
    out = torch.full((out_f, in_f), float("nan"), device=cuda_device, dtype=dtype)
    if r == 0:
        ops.pack_weight(w, out)
        assert torch.equal(out, w.to(dtype))
        return
    A = torch.randn(r, in_f, generator=g).to(cuda_device) * 0.1
    Bm = torch.randn(out_f, r, generator=g).to(cuda_device) * 0.1
    s = 0.37
    ops.pack_weight(w, out, A, Bm, s)
    ref = w.double() + s * (Bm.double() @ A.double())
    mag = w.double().abs() + s * (Bm.double().abs() @ A.double().abs())
    if dtype == torch.float32:
        c = ((out.double() - ref).abs() / (U32 * mag)).max().item()
        print(f"[fwd:pack] f32 r={r}: c={c:.2f}")
        assert c <= PACK_C(r)
    else:
        # one ulp of the rounded fp64 value, beyond what the fp32 sum can lose where W and s B A cancel (|ref| << mag)
        err = ((out.double() - ref.to(dtype).double()).abs() - PACK_C(r) * U32 * mag).clamp_min(0.0) / _ulp(ref, dtype)
        print(f"[fwd:pack] {dname} r={r}: {err.max().item():.2f} ulp from the rounded fp64 value")
        assert err.max().item() <= 1.0


KVNORM_C = 15.0     # c in |v_ip_norm - ||v||| <= c u ||v||: observed 5.8


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("C,Li", [(320, 1), (640, 16), (1280, 5)])
def test_kv_pack_workspaces_and_value_norms(cuda_device, dname, C, Li):
    """The fp32 K / V projections pv_kv_pack_fwd leaves in its workspaces (per element against fp64), and ||V_img|| per
    (sample, head, image token) against the fp64 norm of that same workspace."""
    from photoverse_b200 import _lib
    dtype = DTYPES[dname]
    B, Lt = 3, 77
    case = (f"kv_{C}_{Li}", B, 1, C, Lt, Li, "zero_img")
    _, _, text, img, wkv_t, wkv_i = cross_inputs(*case)
    text, img, wkv_t, wkv_i = (t.to(cuda_device, dtype).contiguous() for t in (text, img, wkv_t, wkv_i))
    d = C // H
    tile = int(_lib.lib().pv_kv_tile_bytes(_code(dtype), C, H, Lt, Li))
    Kp = torch.full((B * H * tile,), 0xFF, device=cuda_device, dtype=torch.uint8)
    Vp = Kp.clone()
    kt = torch.full((B * Lt, 2 * C), float("nan"), device=cuda_device)
    ki = torch.full((B * Li, 2 * C), float("nan"), device=cuda_device)
    vn = torch.full((B, H, Li), float("nan"), device=cuda_device)
    _lib.check(_lib.lib().pv_kv_pack_fwd(_code(dtype), _vp(text), _vp(img), _vp(wkv_t), _vp(wkv_i), _vp(kt), _vp(ki), _vp(Kp),
                                         _vp(Vp), _vp(vn), B, Lt, Li, DC, C, H, _stream()), "pv_kv_pack_fwd")
    fails = []
    for name, ws, tok in (("kv_text", kt, text), ("kv_img", ki, img)):
        tk = tok.double().view(-1, DC)
        wk = wkv_t if name == "kv_text" else wkv_i
        ref = tk @ wk.double().t()
        mag = tk.abs() @ wk.double().abs().t()
        c = ((ws.double() - ref).abs() / (U32 * mag).clamp_min(1e-300)).max().item()
        print(f"[fwd:kvpack] {dname} C{C} Li{Li} {name}: c={c:.2f}")
        if not c <= GEMM_C:
            fails.append(f"{name}: error {c:.1f} u |t||W|^T > {GEMM_C}")
    # the operand tiles, whatever their layout: per (sample, head) the values of K (of V) rounded to the compute dtype
    # and zeros for the padding -- a byte left from the 0xFF poison is a NaN and matches nothing
    for name, img_ in (("Kp", Kp), ("Vp", Vp)):
        part = 0 if name == "Kp" else 1
        vals = torch.cat([kt.view(B, Lt, 2, H, d)[:, :, part], ki.view(B, Li, 2, H, d)[:, :, part]], 1)   # [B, L, H, d]
        vals = vals.transpose(1, 2).reshape(B * H, -1).to(dtype)
        got = img_.view(dtype).view(B * H, -1)
        want = torch.cat([vals, torch.zeros(B * H, got.shape[1] - vals.shape[1], device=cuda_device, dtype=dtype)], 1)
        if not torch.equal(got.sort(1).values, want.sort(1).values):
            fails.append(f"{name}: the tile values are not the rounded {name[0]} of the workspace (or a byte is unwritten)")
    nref = ki.double().view(B, Li, 2, H, d)[:, :, 1].norm(dim=-1).transpose(1, 2)
    cn = ((vn.double() - nref).abs() / (U32 * nref).clamp_min(1e-300)).max().item()
    print(f"[fwd:kvpack] {dname} C{C} Li{Li} v_ip_norm: c={cn:.2f}")
    if not cn <= KVNORM_C:
        fails.append(f"v_ip_norm: error {cn:.1f} u ||v|| > {KVNORM_C}")
    if not torch.equal(vn[B - 1, :, zero_token(Li)], torch.zeros(H, device=cuda_device)):
        fails.append("v_ip_norm of the all-zero image token is not 0")
    assert not fails, "\n".join(fails)


LN_C = 7.0          # c of the fp32 part of the ln_lrelu bound: observed 2.6; of the saved rstd (relative): observed 2.1
LN_MEAN_C = 2.0     # c in |mean - mean64| <= c u mean|x|: observed 0.65


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("cols", [768, 1024])
@pytest.mark.parametrize("rpg", [1, 63, 64, 65])
def test_ln_lrelu_elementwise_row_strided(cuda_device, dname, cols, rpg):
    """LayerNorm + per-group affine + LeakyReLU of the adapter, x and out row-strided views, saved mean / rstd."""
    from photoverse_b200 import ops
    dtype = DTYPES[dname]
    groups = 3
    rows = groups * rpg
    g = torch.Generator().manual_seed(cols + rpg)
    xb = (torch.randn(rows, cols + 24, generator=g) * 2 + 0.3).to(cuda_device)
    x = xb[:, 8:8 + cols]
    gamma = (1 + 0.2 * torch.randn(groups, cols, generator=g)).to(cuda_device)
    beta = (0.3 * torch.randn(groups, cols, generator=g)).to(cuda_device)
    ob = torch.full((rows, cols + 24), 7.0, device=cuda_device, dtype=dtype)
    ob[:, 8:8 + cols] = float("nan")
    out = ob[:, 8:8 + cols]
    fails = []
    for slope in (0.01, 0.2):
        _, mean, rstd = ops.ln_lrelu(x, gamma, beta, out, rows_per_group=rpg, slope=slope, save_stats=True)
        xd = x.double()
        m64 = xd.mean(1)
        r64 = 1.0 / torch.sqrt(xd.var(1, unbiased=False) + 1e-5)
        xhat = (xd - m64[:, None]) * r64[:, None]
        gd, bd = gamma.double().repeat_interleave(rpg, 0), beta.double().repeat_interleave(rpg, 0)
        hh = xhat * gd + bd
        ref = torch.where(hh > 0, hh, slope * hh)
        mag = (xhat.abs() + r64[:, None] * (xd.abs() + m64.abs()[:, None])) * gd.abs() + bd.abs()
        k = torch.where(hh > 0, 1.0, slope)
        c = (((out.double() - ref).abs() - _out_round(ref, dtype)).clamp_min(0.0) / (U32 * k * mag)).max().item()
        cm = ((mean.double() - m64).abs() / (U32 * xd.abs().mean(1))).max().item()
        cr = ((rstd.double() / r64 - 1.0).abs() / U32).max().item()
        print(f"[fwd:ln] {dname} cols={cols} rpg={rpg} slope={slope}: c={c:.2f} mean_c={cm:.2f} rstd_c={cr:.2f}")
        if not (c <= LN_C and cm <= LN_MEAN_C and cr <= LN_C):
            fails.append(f"slope={slope}: c={c:.1f} rstd c={cr:.1f} (bound {LN_C}), mean c={cm:.1f} (bound {LN_MEAN_C})")
    assert torch.equal(ob[:, :8], torch.full((rows, 8), 7.0, device=cuda_device, dtype=dtype))
    assert torch.equal(ob[:, 8 + cols:], torch.full((rows, 16), 7.0, device=cuda_device, dtype=dtype))
    assert not fails, "\n".join(fails)


GROUP_MEAN_C = 8.0   # c in |got - mean| <= u_out |mean| + c u mean|x|: observed 3.25 (fp32, P = 7)


@pytest.mark.gpu
@pytest.mark.parametrize("io", ["f32-f32", "f32-bf16", "f32-f16", "bf16-bf16", "bf16-f32", "f16-f16", "f16-f32"])
@pytest.mark.parametrize("P", [1, 7, 256])
def test_group_mean_into_row_strided_out(cuda_device, io, P):
    from photoverse_b200 import ops
    din, dout = (DTYPES[s] for s in io.split("-"))
    groups, cols = 3, 1024
    g = torch.Generator().manual_seed(P)
    x = (torch.randn(groups, P, cols, generator=g) + 0.5).to(cuda_device, din)
    ob = torch.full((groups, cols + 32), 7.0, device=cuda_device, dtype=dout)
    ob[:, 16:16 + cols] = float("nan")
    out = ob[:, 16:16 + cols]
    ops.group_mean(x, out)
    ref = x.double().mean(1)
    c = (((out.double() - ref).abs() - _out_round(ref, dout)).clamp_min(0.0) / (U32 * x.double().abs().mean(1))).max().item()
    print(f"[fwd:group_mean] {io} P={P}: c={c:.2f}")
    assert torch.isfinite(out.double()).all()
    assert c <= GROUP_MEAN_C
    if P == 1 and din == dout:
        assert torch.equal(out, x[:, 0])
    assert torch.equal(ob[:, :16], torch.full((groups, 16), 7.0, device=cuda_device, dtype=dout))
    assert torch.equal(ob[:, 16 + cols:], torch.full((groups, 16), 7.0, device=cuda_device, dtype=dout))


# ------------------------------------------------------------------------------------------------------------
# §6  switches documented as bit-identical (DESIGN 4.1): attn6_prefetch x attn6_token
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "f16"])
@pytest.mark.parametrize("fuse", [2, 0], ids=["one-launch", "two-launch"])
@pytest.mark.parametrize("B,S,C,Lt,Li", [(2, 300, 320, 77, 5), (1, 1000, 320, 76, 16), (2, 300, 640, 77, 2),
                                         (3, 513, 640, 20, 16)])
def test_attn6_switches_are_bit_identical(cuda_device, dname, fuse, B, S, C, Lt, Li):
    from photoverse_b200 import _lib
    dtype = DTYPES[dname]
    case = (f"sw_{S}_{C}", B, S, C, Lt, Li, "")
    xq, wq, kv, _, _, _ = _cross_operands(case, dtype, cuda_device)
    g = torch.Generator().manual_seed(S)
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(cuda_device, dtype)
    bo = torch.randn(C, generator=g).to(cuda_device)
    runs = {}
    _lib.set_option("fuse_out", fuse)
    try:
        for pre in (1, 0):
            for tok in (1, 0):
                _lib.set_option("attn6_prefetch", pre)
                _lib.set_option("attn6_token", tok)
                runs[(pre, tok)] = _fwd_call(dtype, xq, wq, kv, wo, bo, B, S, C, Lt, Li, 1.0, 1.0)
                assert _all_sync_counters_zero(), f"row-block counters not zero after attn6_prefetch={pre} attn6_token={tok}"
    finally:
        _lib.set_option("attn6_prefetch", 1)
        _lib.set_option("attn6_token", 1)
        _lib.set_option("fuse_out", 1)
    y1, o1, st1, n1 = runs[(1, 1)]
    assert n1 == (1 if fuse == 2 else 2)
    assert torch.isfinite(y1).all() and torch.isfinite(o1).all() and torch.isfinite(st1).all()
    for key, (y, o, st, n) in runs.items():
        assert n == n1
        assert torch.equal(o, o1) and torch.equal(y, y1) and torch.equal(st, st1), f"attn6_prefetch, attn6_token = {key}"


# ------------------------------------------------------------------------------------------------------------
# §7  CPU: the checkers reject small mistakes at the bounds chosen above
# ------------------------------------------------------------------------------------------------------------
def _cpu_cross_case(B=1, S=64, C=320, Lt=76, Li=16):
    """Q rounded to bf16 and fp16, and the fp32 K / V workspaces, on the CPU from cross_inputs."""
    x, wq, text, img, wkv_t, wkv_i = cross_inputs("selftest", B, S, C, Lt, Li, "")
    kt = (text.double().view(-1, DC) @ wkv_t.double().t()).float()
    ki = (img.double().view(-1, DC) @ wkv_i.double().t()).float()
    q = {dt: (x.to(dt).double() @ wq.to(dt).double().t()).to(dt) for dt in (torch.bfloat16, torch.float16)}
    return q, kt, ki


def test_cross_attention_checker_rejects_small_mistakes():
    B, S, C, Lt, Li = 1, 129, 320, 76, 16
    d = C // H
    q, kt32, ki32 = _cpu_cross_case(B, S, C, Lt, Li)
    for dt in (torch.bfloat16, torch.float16):
        bounds = CROSS_BOUNDS[dt]
        kt, ki = kt32.to(dt), ki32.to(dt)
        rt, ri, _ = cross_segments(q[dt], kt, ki, B, Lt, Li)
        for wt, wi in WEIGHTS:
            ref = wt * rt + wi * ri
            # the fp64 reference rounded to the compute dtype, and the kernels' rounding model, pass
            assert not check_cross(ref.to(dt), rt, ri, wt, wi, B, S, d, bounds, "rounded")[1]
            assert not check_cross(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, dt), rt, ri, wt, wi, B, S, d, bounds,
                                   "model")[1]
        wt, wi = 1.3, 0.6

        def fails(got):
            return check_cross(got, rt, ri, wt, wi, B, S, d, bounds, "mutant")[1]

        good = cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, dt)
        assert fails(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, dt, w_scale=(1.0, 1.01))), "image weight x 1.01"
        assert fails(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, dt, w_scale=(1.01, 1.0))), "text weight x 1.01"
        assert fails(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, o_dtype=dt, trunc=True)), "P truncated, l unrounded"
        g = good.clone()
        g[0, 21] = good[0, 22]
        assert fails(g), "query row 21 replaced by row 22"
        g = good.clone()
        g[:, 128:] = cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, dt, w_scale=(1.0, 1.01))[:, 128:]
        assert fails(g), "image weight x 1.01 in the ragged last row tile only"
        g = good.clone().view(B, S, H, d)
        g[:, :, 3] = good.view(B, S, H, d)[:, :, 4]
        assert fails(g.view(B, S, C)), "head 3 taken from head 4"
        kt_drop = kt.view(B, Lt, 2 * C)[:, :Lt - 1].reshape(-1, 2 * C)
        rt_drop, _, _ = cross_segments(q[dt], kt_drop, ki, B, Lt - 1, Li)
        assert fails((wt * rt_drop + wi * ri).to(dt)), "text key 75 dropped"
        ki_drop = ki.view(B, Li, 2 * C)[:, :Li - 1].reshape(-1, 2 * C)
        _, ri_drop, _ = cross_segments(q[dt], kt, ki_drop, B, Lt, Li - 1)
        assert fails((wt * rt + wi * ri_drop).to(dt)), "image key 15 dropped"
        if dt == torch.float16:
            # a bf16 rounding inside an fp16 kernel
            assert fails(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, torch.bfloat16, dt)), "fp16 kernel with P in bf16"
            assert fails(cross_model(q[dt], kt, ki, B, Lt, Li, wt, wi, dt, torch.bfloat16)), "fp16 kernel with a bf16 O drain"


def test_self_attention_checker_rejects_small_mistakes():
    """At the flat bounds: the reference rounded to bf16 and the kernel's rounding model pass; a denominator from the
    unrounded P, one query row from its neighbour and one head from the next head fail."""
    B, S, C = 1, 300, 320
    d = C // H
    SELF_BOUNDS_ = SELF_BOUNDS["flat"]
    g = torch.Generator().manual_seed(4)
    qkv = (torch.randn(B, S, 3 * C, generator=g) * SELF_SCALE["flat"]).bfloat16()
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    ref = self_ref(q, k, v, B, S, C)
    assert not check_self(ref.bfloat16(), ref, B, S, d, SELF_BOUNDS_, "rounded")[1]
    good = self_model(q, k, v, B, S, C)
    assert not check_self(good, ref, B, S, d, SELF_BOUNDS_, "model")[1]
    assert check_self(self_model(q, k, v, B, S, C, bad_denominator=True), ref, B, S, d, SELF_BOUNDS_, "mutant")[1]
    m = good.clone()
    m[0, 100] = good[0, 101]
    assert check_self(m, ref, B, S, d, SELF_BOUNDS_, "mutant")[1]
    m = good.clone().view(B, S, H, d)
    m[:, :, 5] = good.view(B, S, H, d)[:, :, 6]
    assert check_self(m.view(B, S, C), ref, B, S, d, SELF_BOUNDS_, "mutant")[1]
