"""GPU (B200): regional identity masks (diffusers' ``ip_adapter_masks``) -- the native downsample against the restatement
of diffusers' rule, the masked forward of every kernel family and dtype against the fp64 oracle
(tests/ip_mask_reference.py), the bit-identity of an all-ones mask, masked training against autograd through the oracle,
the launch sequence and generation.  Tolerances are those of test_gpu_lora_out.py / test_gpu_backward.py."""
import pytest
import torch

from oracle import cases
from tests.helpers import force_fusion_seed
from tests.ip_mask_reference import clone_with_masked_oracle_processors, downsample, masked_attention
from tests.test_gpu_lora_out import FWD_TOL, REL, _layer, _rel, _trainable, _weights

pytestmark = pytest.mark.gpu

F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64


def _mask(kind, mb, h=64, w=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    if kind == "rand":
        m = torch.rand(mb, 1, h, w, generator=g)
    elif kind == "binary":
        m = torch.zeros(mb, 1, h, w)
        m[..., : w // 2] = 1.0                        # left half: one face of a group photo
        if mb > 1:
            m[1:] = 1.0 - m[1:]
    elif kind == "ones":
        m = torch.ones(mb, 1, h, w)
    else:
        m = torch.zeros(mb, 1, h, w)
    return m


def _sync_words_zero():
    from photoverse_b200 import ops
    torch.cuda.synchronize()
    return all(int(b.abs().sum().item()) == 0 for b in ops._SYNC.values())


# ---- downsample kernel ---------------------------------------------------------------------------------------------
GRIDS = [4096, 1024, 256, 64, 9216, 2304, 576, 144]          # the query grids of 512^2 and 768^2 generation


@pytest.mark.parametrize("mb,h,w", [(1, 64, 64), (3, 64, 64), (1, 96, 64), (1, 64, 100), (3, 512, 384)])
def test_downsample_kernel_matches_reference(cuda_device, mb, h, w):
    from photoverse_b200 import ops
    B = 3
    m = torch.rand(mb, h, w, generator=torch.Generator().manual_seed(h * w + mb))
    m[:, : h // 3] = (m[:, : h // 3] > 0.5).float()            # sharp edges as well as smooth values
    for S in GRIDS:
        got = ops.ip_mask_rows(m.to(cuda_device), B, S)
        ref = downsample(m.double(), B, S)
        err = (got.double().cpu() - ref).abs().max().item()
        assert err <= 1e-6, f"S={S}: max-abs {err}"


# ---- masked forward ------------------------------------------------------------------------------------------------
FWD_SHAPES = [(2, 4096, 320, 5), (2, 1024, 640, 1), (2, 256, 1280, 16), (2, 64, 1280, 5),     # the SD-1.5 attn2 layers
              (3, 200, 320, 5), (2, 100, 640, 16), (1, 520, 640, 1)]                           # ragged, S <= 128


@pytest.mark.parametrize("kind", ["rand", "binary", "ones", "zeros"])
@pytest.mark.parametrize("B,S,C,Li", FWD_SHAPES, ids=[f"B{b}_S{s}_C{c}_Li{li}" for b, s, c, li in FWD_SHAPES])
def test_masked_forward_matches_oracle(cuda_device, B, S, C, Li, kind):
    """bf16 / fp16 (fuse_out 0, 1, 2) and fp32, merged LoRA on q/k/v and out, masks of batch 1 and B; the ws_sync words
    are zero after every call."""
    from photoverse_b200 import _lib
    case = cases.ProcCase(f"mask_{S}_{C}", B=B, S=S, C=C, Li=Li, lora_r=8, seed=300 + S % 97 + Li)
    attn, proc = _layer(case, cuda_device, 4)
    x, text, img = cases.proc_inputs(case, F32)
    w = _weights(case, 4, F64, cuda_device)
    for mb in (1, B):
        mask = _mask(kind, mb, seed=S + mb)
        rows = downsample(mask[:, 0].double(), B, S).to(cuda_device)
        with torch.no_grad():
            y_ref, _ = masked_attention(*(t.to(cuda_device, F64) for t in (x, text, img)), w, 1.0, 1.0, rows)
        for dtype in (BF16, F16, F32):
            for fuse in ((0, 1, 2) if dtype != F32 else (1,)):
                _lib.set_option("fuse_out", fuse)
                try:
                    with torch.no_grad():
                        y = attn(x.to(cuda_device, dtype), encoder_hidden_states=(text.to(cuda_device, dtype),
                                                                                   img.to(cuda_device, dtype)),
                                 ip_adapter_masks=[mask.to(cuda_device)])
                finally:
                    _lib.set_option("fuse_out", 1)
                err = (y.double() - y_ref).abs().max().item()
                assert err <= FWD_TOL[dtype], f"{dtype} fuse_out={fuse} mask batch {mb}: max-abs {err}"
                assert _sync_words_zero()


def test_masked_forward_under_autocast(cuda_device):
    """A float32 model under bf16 autocast computes the masked call in bf16."""
    case = cases.ProcCase("mask_autocast", B=2, S=1024, C=640, Li=5, lora_r=8, seed=331)
    attn, proc = _layer(case, cuda_device, 0)
    x, text, img = cases.proc_inputs(case, F32)
    mask = _mask("rand", 1, 48, 80, seed=3)
    rows = downsample(mask[:, 0].double(), 2, 1024).to(cuda_device)
    with torch.no_grad():
        y_ref, _ = masked_attention(*(t.to(cuda_device, F64) for t in (x, text, img)), _weights(case, 0, F64, cuda_device),
                                    1.0, 1.0, rows)
        with torch.autocast("cuda", dtype=BF16):
            y = attn(x.to(cuda_device), encoder_hidden_states=(text.to(cuda_device), img.to(cuda_device)),
                     ip_adapter_masks=[mask.to(cuda_device)])
    assert y.dtype == BF16
    assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[BF16]


CORE_SHAPES = [(2, 4096, 320, 8), (2, 1024, 640, 8), (2, 256, 1280, 8), (2, 100, 640, 8), (2, 300, 640, 16)]


@pytest.mark.parametrize("B,S,C,H", CORE_SHAPES, ids=[f"S{s}_C{c}_H{h}" for _, s, c, h in CORE_SHAPES])
def test_all_ones_and_null_are_bit_identical(cuda_device, B, S, C, H):
    """Per family and dtype: an all-ones row weight and the NULL pointer through the masked entry points give exactly
    the unmasked entry points' O, Y and statistics: pv_attn6.cu (head_dim 40 / 80), pv_attn4.cu (head_dim 160, and
    head_dim 40 at C = 640), pv_attn3.cu (S <= 128) and the fp32 SIMT kernel."""
    from photoverse_b200 import _lib, ops
    lib = _lib.lib()
    g = torch.Generator().manual_seed(S + C)
    for dtype in (BF16, F16, F32):
        for Li, Lt in ((1, 77), (5, 77), (16, 40)):
            x = (torch.randn(B, S, C, generator=g) * 0.5).to(cuda_device, dtype)
            wq = (torch.randn(C, C, generator=g) / C ** 0.5).to(cuda_device, dtype)
            wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(cuda_device, dtype)
            bo = torch.randn(C, generator=g).to(cuda_device)
            text = torch.randn(B, Lt, 768, generator=g).to(cuda_device, dtype)
            img = torch.randn(B, Li, 768, generator=g).to(cuda_device, dtype)
            wkv = [(torch.randn(2 * C, 768, generator=g) / 28).to(cuda_device, dtype) for _ in range(2)]
            kv = ops.kv_pack(text, img, wkv[0], wkv[1], H)
            ones = torch.ones(B, S, device=cuda_device)
            for wt, wi in ((1.0, 1.0), (2.0, 0.0), (0.0, 2.0)):
                outs = []
                for arm, rw in enumerate((None, None, ones)):
                    if arm == 0:
                        y, o = torch.empty_like(x), torch.empty_like(x)
                        q = torch.empty(B, S, C, device=cuda_device) if dtype == F32 else None
                        st = torch.empty(B, H, S, 4, device=cuda_device)
                        sync = ops._sync_words(B, S, x.device) if dtype != F32 else None
                        _lib.check(lib.pv_dual_attn_fwd(ops._dt(x), ops._ptr(x), ops._ptr(wq), ops._ptr(kv.Kp),
                                                        ops._ptr(kv.Vp), ops._ptr(wo), ops._ptr(bo), ops._ptr(y),
                                                        ops._ptr(q), ops._ptr(o), ops._ptr(st), ops._ptr(sync), B, S, C,
                                                        H, Lt, Li, wt, wi, ops._stream()))
                        oc, stc = torch.empty_like(x), torch.empty(B, H, S, 4, device=cuda_device)
                        xq = x if dtype != F32 else q
                        _lib.check(lib.pv_dual_attn_core_fwd(ops._dt(x), ops._ptr(xq), ops._ptr(wq), ops._ptr(kv.Kp),
                                                             ops._ptr(kv.Vp), ops._ptr(oc), ops._ptr(stc), B, S, C, H, Lt,
                                                             Li, wt, wi, ops._stream()))
                    else:
                        y, o, st, q = ops.dual_attn(x, wq, kv, wo, bo, wt, wi, want_stats=True, img_row_weight=rw)
                        xq = x if dtype != F32 else q
                        oc, stc = ops.dual_attn_core(xq, wq, kv, wt, wi, want_stats=True, img_row_weight=rw)
                    outs.append((y, o, st, oc, stc))
                for arm in (1, 2):
                    for name, a, b in zip(("Y", "O", "stats", "core O", "core stats"), outs[0], outs[arm]):
                        assert torch.equal(a, b), f"{dtype} Li={Li} ({wt},{wi}) {'NULL' if arm == 1 else 'ones'}: {name}"
            assert _sync_words_zero()


def test_all_zeros_mask_is_the_text_branch(cuda_device):
    """A zero mask matches w_img = 0 within tolerance (bf16 and fp32)."""
    case = cases.ProcCase("mask_zeros", B=2, S=1024, C=640, Li=5, seed=341)
    attn, proc = _layer(case, cuda_device, 0)
    x, text, img = cases.proc_inputs(case, F32)
    with torch.no_grad():
        from oracle.processor_oracle import dual_branch_attention
        y_ref, _ = dual_branch_attention(*(t.to(cuda_device, F64) for t in (x, text, img)),
                                         _weights(case, 0, F64, cuda_device), 1.0, 0.0)
        for dtype in (BF16, F32):
            y = attn(x.to(cuda_device, dtype), encoder_hidden_states=(text.to(cuda_device, dtype),
                                                                       img.to(cuda_device, dtype)),
                     ip_adapter_masks=[torch.zeros(1, 1, 32, 32, device=cuda_device)])
            assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[dtype]


def test_launch_count_equals_unmasked_once_cached(cuda_device):
    from photoverse_b200 import _lib
    case = cases.ProcCase("mask_launch", B=2, S=4096, C=320, Li=5, seed=351)
    attn, proc = _layer(case, cuda_device, 0)
    x, text, img = (t.to(cuda_device, BF16) for t in cases.proc_inputs(case, F32))
    mask = [_mask("rand", 1, seed=5).to(cuda_device)]
    with torch.no_grad():
        attn(x, encoder_hidden_states=(text, img), ip_adapter_masks=mask)        # fills the row-weight cache
        n0 = _lib.launch_count()
        attn(x, encoder_hidden_states=(text, img))
        n1 = _lib.launch_count()
        attn(x, encoder_hidden_states=(text, img), ip_adapter_masks=mask)
        n2 = _lib.launch_count()
    assert n2 - n1 == n1 - n0 > 0


# ---- masked training -----------------------------------------------------------------------------------------------
def _oracle_grads(w, x, text, img, gy, gv, wt, wi, rows, drop=None):
    dev, dt = w.to_q.device, w.to_q.dtype
    leaves = {k: t.to(dev, dt).clone().requires_grad_(True) for k, t in (("x", x), ("text", text), ("img", img))}
    w.to_k_ip.requires_grad_(True)
    w.to_v_ip.requires_grad_(True)
    for lw in w.lora.values():
        lw.A.requires_grad_(True)
        lw.B.requires_grad_(True)
    y, vn = masked_attention(leaves["x"], leaves["text"], leaves["img"], w, wt, wi, rows, drop)
    ((y * gy.to(dev, dt)).sum() + (vn.squeeze(-1) * gv.to(dev, dt)).sum()).backward()
    out = {k: v.grad for k, v in leaves.items()}
    out["to_k_ip"], out["to_v_ip"] = w.to_k_ip.grad, w.to_v_ip.grad
    for name, lw in w.lora.items():
        out[name + ".A"], out[name + ".B"] = lw.A.grad, lw.B.grad
    return y.detach(), out


def _masked_train_call(attn, proc, case, dtype, dev, gy, gv, mask, cuda_seed=None):
    x, text, img = cases.proc_inputs(case, F32)
    xd, td, im = (t.to(dev, dtype).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)
    if cuda_seed is not None:
        torch.cuda.manual_seed(cuda_seed)
    with torch.enable_grad():
        y = attn(xd, encoder_hidden_states=(td, im), ip_adapter_masks=[mask.to(dev)])
        assert proc.last_fusion == (case.w_text, case.w_img)
        ((y.float() * gy.to(dev)).sum() + (proc.to_v_ip_norm.float().squeeze(-1) * gv.to(dev)).sum()).backward()
    return y.detach(), {"x": xd.grad, "text": td.grad, "img": im.grad}


def _check(got, ref, tol):
    for k, r in ref.items():
        if r is None or r.abs().max() == 0:
            assert got[k] is None or got[k].abs().max().item() <= 1e-6, k
            continue
        assert got[k] is not None, f"no gradient for {k}"
        e = _rel(got[k], r)
        assert e <= tol, f"{k}: relative error {e:.3e} > {tol}"


TRAIN_CASES = [
    cases.ProcCase("mask_bwd_c320_s4096", B=16, S=4096, C=320, Li=5, lora_r=8, seed=361),             # tcgen05 backward
    cases.ProcCase("mask_bwd_c320_textonly", B=4, S=4096, C=320, Li=5, lora_r=8, w_text=2.0, w_img=0.0, seed=362),
    cases.ProcCase("mask_bwd_c320_imgonly", B=4, S=4096, C=320, Li=1, lora_r=8, w_text=0.0, w_img=2.0, seed=363),
    cases.ProcCase("mask_bwd_c1280_s256", B=2, S=256, C=1280, Li=16, lora_r=8, seed=364),           # head_dim-160 mma.sync
    cases.ProcCase("mask_bwd_c1280_s256_imgonly", B=2, S=256, C=1280, Li=5, lora_r=8, w_text=0.0, w_img=2.0, seed=365),
    cases.ProcCase("mask_bwd_c640_s200", B=2, S=200, C=640, Li=5, lora_r=8, seed=366),
]


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", TRAIN_CASES, ids=lambda c: c.name)
def test_masked_training_matches_oracle_autograd(cuda_device, case, dtype):
    """Forward and every gradient (x, contexts, to_k_ip / to_v_ip, LoRA factors of q, k, v and out) in all three fusion
    branches; fp32 runs the SIMT backward.  Two runs are bit-identical."""
    if dtype == F32 and case.B * case.S > 16384:
        pytest.skip("the fp32 SIMT arm runs the smaller shapes")
    mask = _mask("rand", 1, 48, 64, seed=case.seed)
    rows = downsample(mask[:, 0].double(), case.B, case.S).to(cuda_device)
    g = torch.Generator().manual_seed(case.seed)
    gy, gv = torch.randn(case.B, case.S, case.C, generator=g), torch.randn(case.B, case.H, case.Li, generator=g)
    runs = []
    for _ in range(2):
        attn, proc = _layer(case, cuda_device, 4)
        trainable = _trainable(attn, proc)
        y, got = _masked_train_call(attn, proc, case, dtype, cuda_device, gy, gv, mask)
        got.update({k: p.grad for k, p in trainable.items()})
        runs.append((y, got))
    for k, t in runs[0][1].items():
        assert (t is None and runs[1][1][k] is None) or torch.equal(t, runs[1][1][k]), f"not deterministic: {k}"
    assert torch.equal(runs[0][0], runs[1][0])
    y, got = runs[0]
    x, text, img = cases.proc_inputs(case, F32)
    y_ref, ref = _oracle_grads(_weights(case, 4, F64, cuda_device), x, text, img, gy, gv, case.w_text, case.w_img, rows)
    assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[dtype]
    _check(got, ref, REL[dtype])


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
def test_masked_lora_dropout_matches_oracle(cuda_device, dtype):
    """LoRA-dropout path (p = 0.1 on q, k, v, out) with a mask: keep-masks re-drawn in the order q, k, v, out."""
    p_drop = 0.1
    case = cases.ProcCase("mask_drop", B=2, S=1024, C=640, Li=5, lora_r=8, seed=371)
    attn, proc = _layer(case, cuda_device, 4)
    for name in ("to_q", "to_k", "to_v"):
        getattr(attn, name).lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.to_out[0].lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.train()
    trainable = _trainable(attn, proc)
    mask = _mask("binary", 2, 64, 64)
    rows = downsample(mask[:, 0].double(), case.B, case.S).to(cuda_device)
    g = torch.Generator().manual_seed(case.seed)
    gy, gv = torch.randn(case.B, case.S, case.C, generator=g), torch.randn(case.B, case.H, case.Li, generator=g)
    y, got = _masked_train_call(attn, proc, case, dtype, cuda_device, gy, gv, mask, cuda_seed=2000)
    got.update({k: p.grad for k, p in trainable.items()})
    x, text, img = cases.proc_inputs(case, F32)
    torch.cuda.manual_seed(2000)
    drop = {}
    for name, shape in (("to_q", x.shape), ("to_k", text.shape), ("to_v", text.shape), ("to_out", x.shape)):
        _, keep = torch.native_dropout(torch.zeros(shape, device=cuda_device, dtype=dtype), p_drop, True)
        drop[name] = (keep, p_drop)
    y_ref, ref = _oracle_grads(_weights(case, 4, F64, cuda_device), x, text, img, gy, gv, 1.0, 1.0, rows, drop)
    assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[dtype]
    _check(got, ref, REL[dtype])


# ---- generation ----------------------------------------------------------------------------------------------------
def test_generation_with_a_mask(cuda_device):
    """run_generation (K/V cache and CUDA graph on, batched CFG at guidance 7.5) with a mask against the masked oracle
    arm; an all-ones mask gives the unmasked latents bit for bit; GenerationEngine with the mask as a static input."""
    from oracle.host_reference import clone_adapter_as_oracle
    from photoverse_b200.host.pipeline import GenerationEngine, run_generation, synthetic_inputs
    from tests.test_gpu_pipeline import _cos, _models
    unet, ia, ta = _models(cuda_device, BF16)
    inp = synthetic_inputs(2, 64, seed=21, device=cuda_device, dtype=BF16)
    mask = [_mask("binary", 2, 64, 64).to(cuda_device)]
    lat = run_generation(unet, ia, ta, inp, num_steps=50, guidance_scale=7.5, mode="batched", ip_adapter_masks=mask)
    ref_unet = clone_with_masked_oracle_processors(unet)
    ref_ia, ref_ta = clone_adapter_as_oracle(ia, cuda_device, BF16), clone_adapter_as_oracle(ta, cuda_device, BF16)
    ref = run_generation(ref_unet, ref_ia, ref_ta, inp, num_steps=50, guidance_scale=7.5, mode="two_call",
                         use_cuda_graph=False, kv_cache=False, ip_adapter_masks=mask)
    plain = run_generation(unet, ia, ta, inp, num_steps=50, guidance_scale=7.5, mode="batched")
    c, c_plain = _cos(lat, ref), _cos(lat, plain)
    print(f"masked generation: final-latent cosine vs the masked oracle arm {c:.6f}, vs unmasked {c_plain:.6f}")
    assert c >= 0.999
    assert c_plain < 0.999                                   # the mask changes the result
    ones = run_generation(unet, ia, ta, inp, num_steps=50, guidance_scale=7.5, mode="batched",
                          ip_adapter_masks=[torch.ones(1, 1, 64, 64, device=cuda_device)])
    assert torch.equal(ones, plain)
    # the engine: one captured evaluation, the static mask refreshed by load_inputs
    eng_in = synthetic_inputs(2, 32, seed=22, device=cuda_device, dtype=BF16)
    m1, m2 = _mask("rand", 1, 32, 32, seed=1), _mask("binary", 1, 32, 32)
    eng = GenerationEngine(unet, ia, ta, batch=2, latent=32, num_steps=10, guidance_scale=7.5, dtype=BF16,
                           device=cuda_device, ip_mask_shape=(32, 32))
    res = []
    for m in (m1, m2, m1):
        eng.load_inputs(eng_in, ip_mask=m.to(cuda_device))
        res.append(eng.generate().clone())
    eng.close()
    assert torch.equal(res[0], res[2]) and not torch.equal(res[0], res[1])
    for m, r in ((m1, res[0]), (m2, res[1])):
        want = run_generation(unet, ia, ta, eng_in, num_steps=10, guidance_scale=7.5, mode="batched",
                              use_cuda_graph=False, ip_adapter_masks=[m.to(cuda_device)])
        assert _cos(r, want) >= 0.9999
