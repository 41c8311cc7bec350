"""GPU (B200): float32 models under torch.autocast (DESIGN.md 4.9) -- the processor, the adapters, the training step and
the generation loop compute in the autocast dtype, through the 16-bit kernels and the pv_convert_fwd conversions.

With parameters that are exactly representable in bf16 (and fp16), a float32 layer under autocast packs the same weights as
its ``.to(bfloat16)`` copy, so its outputs must be bit-identical to that copy's on ``X.to(bfloat16)``, and its native launch
count must be that copy's plus the conversions: neither the fp32 SIMT path nor a torch cast may run."""
import copy

import pytest
import torch

from oracle import cases
from tests.helpers import build_product_layer, force_fusion_seed

pytestmark = pytest.mark.gpu

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
_CODE = {F32: 0, BF16: 1, F16: 2}


def _representable(module):
    """Round every parameter to a value exact in both bf16 and fp16."""
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(p.to(BF16).to(F16).float())


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _assert_same_conversion(got, want):
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan)
    assert torch.equal(_bits(got)[~nan], _bits(want)[~nan])


# ---------------------------------------------------------------------------------------------------------------------
# pv_convert_fwd
# ---------------------------------------------------------------------------------------------------------------------
def _source(dtype, n, device):
    g = torch.Generator().manual_seed(n)
    if dtype == F32:
        special = torch.tensor([0.0, -0.0, 1e-40, -3e-39, 1.4e-45, 6e-8, 3e-5, -6.1e-5, 65504.0, 65519.0, 65520.0, 1e6,
                                -1e6, 3.0e38, float("inf"), float("-inf"), float("nan"), 1.00390625, 1.01171875, -2.5])
        bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=g, dtype=torch.int64).to(torch.int32).view(F32)
        normal = torch.randn(n, generator=g) * 10.0 ** torch.randint(-6, 6, (n,), generator=g).float()
        x = torch.where(torch.arange(n) % 2 == 0, bits, normal)
    else:
        special = torch.tensor([0.0, -0.0, 6e-8, 1e-40, float("inf"), float("-inf"), float("nan"), 1.0, -2.0]).to(dtype)
        x = torch.randint(-2 ** 15, 2 ** 15, (n,), generator=g, dtype=torch.int32).to(torch.int16).view(dtype)
    k = min(n, special.numel())
    x[:k] = special[:k]
    return x.to(device)


@pytest.mark.parametrize("src_off,dst_off", [(0, 0), (1, 0), (0, 1), (1, 1), (3, 3)])
@pytest.mark.parametrize("n", [1, 7, 8, 4097])
@pytest.mark.parametrize("in_dt,out_dt", [(F32, BF16), (F32, F16), (BF16, F32), (F16, F32)], ids=str)
def test_convert_bit_identical_to_tensor_to(cuda_device, in_dt, out_dt, n, src_off, dst_off):
    from photoverse_b200 import _lib, ops
    base = _source(in_dt, n + src_off, cuda_device)
    src = base[src_off:]
    want = src.to(out_dt)
    out_base = torch.full((n + dst_off,), 7, device=cuda_device, dtype=out_dt)
    dst = out_base[dst_off:]
    n0 = _lib.launch_count()
    _lib.check(_lib.lib().pv_convert_fwd(_CODE[in_dt], _CODE[out_dt], src.data_ptr(), dst.data_ptr(), n,
                                         torch.cuda.current_stream().cuda_stream), "pv_convert_fwd")
    assert _lib.launch_count() - n0 == 1
    _assert_same_conversion(dst, want)
    assert (out_base[:dst_off] == 7).all()
    _assert_same_conversion(ops.convert(src.view(1, n), out_dt), want.view(1, n))


def test_convert_large_and_fp16_overflow(cuda_device):
    from photoverse_b200 import ops
    x = torch.randn(3 * 1024 * 1024 + 5, device=cuda_device) * 3e4
    for dt in (BF16, F16):
        y = ops.convert(x, dt)
        _assert_same_conversion(y, x.to(dt))
        _assert_same_conversion(ops.convert(y, F32), y.float())
    assert torch.isinf(ops.convert(x, F16)).any()


# ---------------------------------------------------------------------------------------------------------------------
# processor
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = [(2, 4096, 320, 1), (2, 1024, 640, 5), (2, 256, 1280, 16), (2, 64, 1280, 5), (3, 200, 320, 16)]
SHAPE_IDS = [f"B{b}_S{s}_C{c}_Li{li}" for b, s, c, li in SHAPES]


def _layers(shape, device, half=BF16, seed=0):
    B, S, C, Li = shape
    case = cases.ProcCase(f"ac_{S}_{C}", B=B, S=S, C=C, Li=Li, lora_r=4, seed=40 + Li + seed)
    attn, proc = build_product_layer(case, device)
    _representable(attn)
    attn16 = copy.deepcopy(attn).to(half)
    x, text, img = (t.to(device) for t in cases.proc_inputs(case, F32))
    return case, (attn, proc), (attn16, attn16.processor), (x, text, img)


def _launches(fn):
    from photoverse_b200 import _lib
    fn()                                            # packs the weights
    n0 = _lib.launch_count()
    out = fn()
    return out, _lib.launch_count() - n0


@pytest.mark.parametrize("half", [BF16, F16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_processor_autocast_bit_identical_to_16bit_layer(cuda_device, shape, half):
    _, (attn, proc), (attn16, proc16), (x, text, img) = _layers(shape, cuda_device, half)
    with torch.no_grad():
        y16, n16 = _launches(lambda: attn16(x.to(half), encoder_hidden_states=(text.to(half), img.to(half))))
        vn16 = proc16.to_v_ip_norm
        with torch.autocast("cuda", dtype=half):
            y, n = _launches(lambda: attn(x, encoder_hidden_states=(text, img)))
        vn = proc.to_v_ip_norm
    assert y.dtype == half and torch.equal(y, y16)
    assert n == n16 + 3, (n, n16)                  # + the conversions of X, text and image tokens
    assert vn.dtype == F32 and torch.equal(vn.to(half), vn16)


@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_processor_autocast_grad_matches_bf16_layer(cuda_device, shape):
    case, (attn, proc), (attn16, proc16), (x, text, img) = _layers(shape, cuda_device)

    def trainable(a):
        a.requires_grad_(False)
        ps = {n: p for n, p in a.named_parameters() if "lora_" in n or "to_k_ip" in n or "to_v_ip" in n}
        for p in ps.values():
            p.requires_grad_(True)
        return ps

    ps32, ps16 = trainable(attn), trainable(attn16)
    g = torch.Generator().manual_seed(case.seed)
    dy = torch.randn(case.B, case.S, case.C, generator=g).to(cuda_device, BF16)
    dvn = torch.randn(case.B, case.H, case.Li, 1, generator=g).to(cuda_device, BF16)
    x32, t32 = x.clone().requires_grad_(True), text.clone().requires_grad_(True)
    x16, t16 = x.to(BF16).requires_grad_(True), text.to(BF16).requires_grad_(True)
    force_fusion_seed(1.0, 1.0)
    y16 = attn16(x16, encoder_hidden_states=(t16, img.to(BF16)))
    torch.autograd.backward([y16, proc16.to_v_ip_norm], [dy, dvn])
    force_fusion_seed(1.0, 1.0)
    with torch.autocast("cuda", dtype=BF16):
        y = attn(x32, encoder_hidden_states=(t32, img))
        vn = proc.to_v_ip_norm
    torch.autograd.backward([y, vn], [dy, dvn.float()])
    assert proc.last_fusion == proc16.last_fusion == (1.0, 1.0)
    assert y.dtype == BF16 and torch.equal(y, y16)
    assert x32.grad.dtype == F32 and torch.equal(x32.grad, x16.grad.float())
    assert t32.grad.dtype == F32 and torch.equal(t32.grad, t16.grad.float())
    assert set(ps32) == set(ps16) and len(ps32) == 8
    for n, p in ps32.items():
        assert p.dtype == F32 and p.grad is not None and p.grad.dtype == F32, n
        assert torch.equal(p.grad.to(BF16), ps16[n].grad), n


@pytest.mark.parametrize("case", [
    cases.ProcCase("ac_drop_c320", B=2, S=200, C=320, Li=5, lora_r=8, seed=76),
    cases.ProcCase("ac_drop_c1280", B=1, S=64, C=1280, Li=3, lora_r=16, seed=78),
], ids=lambda c: c.name)
def test_processor_autocast_lora_dropout_matches_oracle(cuda_device, case):
    """LoRA dropout p = 0.1 under bf16 autocast (the unmerged-weight path packed from the float32 masters) against the
    fp64 oracle with the keep-masks re-drawn from the same CUDA seed, at the bf16 tolerance of test_gpu_backward."""
    from tests.test_gpu_backward import REL, _oracle_grads, _rel
    p_drop = 0.1
    attn, proc = build_product_layer(case, cuda_device)
    for name in ("to_q", "to_k", "to_v"):
        getattr(attn, name).lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.train()
    attn.requires_grad_(False)
    trainable = {"to_k_ip": proc.to_k_ip[0].weight, "to_v_ip": proc.to_v_ip[0].weight}
    for name in ("to_q", "to_k", "to_v"):
        m = getattr(attn, name)
        trainable[name + ".A"] = m.lora_A["default"].weight
        trainable[name + ".B"] = m.lora_B["default"].weight
    for p in trainable.values():
        p.requires_grad_(True)
    x, text, img = cases.proc_inputs(case, F32)
    g = torch.Generator().manual_seed(case.seed)
    gy = torch.randn(case.B, case.S, case.C, generator=g)
    gv = torch.randn(case.B, case.H, case.Li, generator=g)
    xd, td, im = (t.to(cuda_device).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)
    torch.cuda.manual_seed(1000 + case.seed)
    with torch.autocast("cuda", dtype=BF16):
        y = attn(xd, encoder_hidden_states=(td, im))
        vn = proc.to_v_ip_norm
        loss = (y.float() * gy.to(cuda_device)).sum() + (vn.float().squeeze(-1) * gv.to(cuda_device)).sum()
    loss.backward()
    assert y.dtype == BF16
    torch.cuda.manual_seed(1000 + case.seed)
    drop = {}
    for name, t in (("to_q", xd), ("to_k", td), ("to_v", td)):     # the masks are drawn on the bf16 activations
        _, mask = torch.native_dropout(t.detach().to(BF16), p_drop, True)
        drop[name] = (mask.cpu(), p_drop)
    y_ref, _, ref = _oracle_grads(case, x, text, img, gy, gv, case.w_text, case.w_img, drop)
    assert (y.detach().float().cpu() - y_ref.float()).abs().max().item() <= 2e-2
    got = {"x": xd.grad, "text": td.grad, "img": im.grad}
    got.update({k: p.grad for k, p in trainable.items()})
    for k, r in ref.items():
        assert got[k] is not None and got[k].dtype == F32, k
        e = _rel(got[k], r)
        assert e <= REL[BF16], f"{k}: relative error {e:.3e} > {REL[BF16]}"


def test_processor_fp16_autocast_grad_mode_is_the_float32_path(cuda_device):
    case, (attn, proc), _, (x, text, img) = _layers((2, 256, 640, 5), cuda_device)
    attn.requires_grad_(False)
    ps = [p for n, p in attn.named_parameters() if "lora_" in n or "_ip" in n]
    for p in ps:
        p.requires_grad_(True)
    dy = torch.randn(case.B, case.S, case.C, device=cuda_device)
    res = []
    for autocast in (False, True):
        xg = x.clone().requires_grad_(True)
        for p in ps:
            p.grad = None
        force_fusion_seed(1.0, 1.0)
        with torch.autocast("cuda", dtype=F16, enabled=autocast):
            y = attn(xg, encoder_hidden_states=(text, img))
            vn = proc.to_v_ip_norm
        torch.autograd.backward([y, vn], [dy, torch.ones_like(vn)])
        res.append([y.detach(), vn.detach(), xg.grad] + [p.grad.clone() for p in ps])
    for a, b in zip(*res):
        assert a.dtype == F32 and torch.equal(a, b)


def test_processor_autocast_kv_cache(cuda_device):
    """Keyed on the caller's context tensors: the cache stops growing after the first call, and a cached call launches
    the bf16 layer's cached call plus the conversion of X."""
    _, (attn, proc), (attn16, proc16), (x, text, img) = _layers((2, 1024, 320, 5), cuda_device)
    t16, i16, x16 = text.to(BF16), img.to(BF16), x.to(BF16)
    with torch.no_grad():
        with torch.autocast("cuda", dtype=BF16):
            y_uncached = attn(x, encoder_hidden_states=(text, img))
        proc.enable_kv_cache(True)
        proc16.enable_kv_cache(True)
        _, n16 = _launches(lambda: attn16(x16, encoder_hidden_states=(t16, i16)))
        with torch.autocast("cuda", dtype=BF16):
            attn(x, encoder_hidden_states=(text, img))
            size = len(proc._kv_cache)
            y, n = _launches(lambda: attn(x, encoder_hidden_states=(text, img)))
            attn(x, encoder_hidden_states=(text, img))
        assert len(proc._kv_cache) == size == 1
        proc.enable_kv_cache(False)
        proc16.enable_kv_cache(False)
    assert n == n16 + 1, (n, n16)
    assert torch.equal(y, y_uncached)


# ---------------------------------------------------------------------------------------------------------------------
# adapters
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c for c in cases.ADAPTER_CASES if c.token_index in (0, "full")], ids=lambda c: c.name)
def test_adapter_autocast_matches_bf16_adapter(cuda_device, case):
    from oracle import adapter_oracle
    from photoverse_b200 import PhotoVerseAdapter
    ad = PhotoVerseAdapter(num_tokens=case.T)
    ad.load_state_dict(adapter_oracle.make_state_dict(case.T, case.seed), strict=True)
    ad.to(cuda_device)
    _representable(ad)
    ad16 = copy.deepcopy(ad).to(BF16)
    embs = [e.to(cuda_device) for e in cases.adapter_inputs(case)]
    embs16 = [e.to(BF16) for e in embs]
    with torch.no_grad():
        y16 = ad16(embs16, token_index=case.token_index)
        with torch.autocast("cuda", dtype=BF16):
            y = ad(embs, token_index=case.token_index)
    assert y.dtype == BF16 and torch.equal(y, y16)
    dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(1)).to(cuda_device, BF16)
    ad16(embs16, token_index=case.token_index).backward(dy)
    with torch.autocast("cuda", dtype=BF16):
        y = ad(embs, token_index=case.token_index)
    y.backward(dy)
    got = dict(ad.named_parameters())
    n_grads = 0
    for n, p16 in ad16.named_parameters():
        if p16.grad is None:
            assert got[n].grad is None, n
            continue
        assert got[n].grad.dtype == F32 and torch.equal(got[n].grad.to(BF16), p16.grad), n
        n_grads += 1
    assert n_grads > 0


# ---------------------------------------------------------------------------------------------------------------------
# training step and generation of a float32 UNet
# ---------------------------------------------------------------------------------------------------------------------
def _all_branches_seed(n_layers):
    """A CPU seed whose next ``n_layers`` draws keep both branches of every layer (every trainable tensor gets a gradient)."""
    for s in range(100000):
        torch.manual_seed(s)
        if all(1 / 3 <= torch.rand(1).item() <= 2 / 3 for _ in range(n_layers)):
            return s
    raise RuntimeError("no seed found")


@pytest.mark.parametrize("fused", [True, False], ids=["fused-epilogues", "stock-epilogues"])
def test_trainer_autocast_bf16_float32_unet(cuda_device, fused):
    """``Trainer(autocast_dtype=bfloat16)`` over a float32 UNet: parameters and gradients stay float32, gradients match
    the fp32 oracle arm at test_gpu_train's bf16 tolerance, and one step moves every trainable tensor.  Stock epilogues
    hand the processors float32 hidden states (nn.LayerNorm under autocast), as diffusers' blocks do."""
    from oracle import adapter_oracle
    from oracle.host_reference import clone_with_oracle_processors
    from photoverse_b200.host.parallel import trainable_named_parameters
    from photoverse_b200.host.train_step import Trainer, synthetic_train_batch
    from photoverse_b200.unet import get_visual_cross_attention_values_norm
    from tests.test_gpu_train import _build, _rel
    unet, ia, ta = _build(cuda_device, F32)
    unet.set_fused_epilogues(fused)
    ref_unet = clone_with_oracle_processors(unet)
    b = synthetic_train_batch(2, latent=16, seed=3, device=cuda_device, dtype=F32)
    tr = Trainer(unet, ia, ta, lr=1e-5, autocast_dtype=BF16)
    named = trainable_named_parameters(unet, ia, ta)
    seed = _all_branches_seed(4)
    torch.manual_seed(seed)
    with torch.enable_grad(), torch.autocast("cuda", dtype=BF16, cache_enabled=False):
        loss, _ = tr.loss(b)
    loss.backward()
    assert all(tr.expected_gradients())
    got = {n: p.grad.detach().clone() for n, p in named}
    # oracle arm in fp32 on the inputs as the reference's first autocast'd matmuls read them, rounded to bf16 (as
    # test_gpu_train's bf16 arm feeds its oracle); the regression target stays float32
    r16 = lambda t: t.to(BF16).float()
    torch.manual_seed(seed)
    with torch.enable_grad():
        emb = [r16(e) for e in b.clip_hidden]
        concept = adapter_oracle.adapter_forward(emb, dict(ta.named_parameters()), None)
        img_tokens = adapter_oracle.adapter_forward(emb, dict(ia.named_parameters()), None)
        pred = ref_unet(r16(b.noisy_latents), b.timesteps, encoder_hidden_states=(r16(b.text), img_tokens)).sample
        l_vis = get_visual_cross_attention_values_norm(ref_unet).mean()
        ref_loss = torch.nn.functional.mse_loss(pred, b.noise) + 0.01 * concept.abs().mean() + 0.001 * l_vis
    for p in ia.parameters():
        p.grad = None
    for p in ta.parameters():
        p.grad = None
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 3e-2 * abs(ref_loss.item())
    ref_named = trainable_named_parameters(ref_unet, ia, ta)
    checked = 0
    for (n, p), (n_ref, p_ref) in zip(named, ref_named):
        assert n == n_ref and p.dtype == F32 and got[n].dtype == F32, n
        if p_ref.grad is None or p_ref.grad.abs().max() == 0:
            continue
        e = _rel(got[n], p_ref.grad)
        assert e <= 1.0e-1, f"{n}: relative error {e:.3e}"
        checked += 1
    assert checked > 100
    before = {n: p.detach().clone() for n, p in named}
    torch.manual_seed(seed)
    loss, _ = tr.step(b)
    assert torch.isfinite(loss)
    for n, p in named:
        assert p.dtype == F32 and not torch.equal(p, before[n]), n


def test_float32_unet_generation_under_bf16_autocast(cuda_device):
    """A float32 UNet through run_generation (CUDA graph + K/V cache) and the GenerationEngine with
    ``autocast_dtype=bfloat16`` vs the oracle-processor arm under the same autocast: final-latent cosine >= 0.999."""
    from tests.test_gpu_pipeline import _cos, _models
    from oracle.host_reference import clone_adapter_as_oracle, clone_with_oracle_processors
    from photoverse_b200.host.pipeline import GenerationEngine, run_generation, synthetic_inputs
    unet, ia, ta = _models(cuda_device, F32)
    ref_unet = clone_with_oracle_processors(unet)
    ref_ia, ref_ta = clone_adapter_as_oracle(ia, cuda_device, F32), clone_adapter_as_oracle(ta, cuda_device, F32)
    inp = synthetic_inputs(2, 32, seed=21, device=cuda_device, dtype=F32)
    lat = run_generation(unet, ia, ta, inp, num_steps=20, mode="batched", use_cuda_graph=True, kv_cache=True,
                         autocast_dtype=BF16)
    ref = run_generation(ref_unet, ref_ia, ref_ta, inp, num_steps=20, mode="two_call", use_cuda_graph=False, kv_cache=False,
                         autocast_dtype=BF16)
    assert lat.dtype == F32 and torch.isfinite(lat).all()
    c = _cos(lat, ref)
    eng = GenerationEngine(unet, ia, ta, batch=2, latent=32, num_steps=20, dtype=F32, device=cuda_device,
                           autocast_dtype=BF16)
    eng.load_inputs(inp)
    e = eng.generate().clone()
    eng.close()
    ce = _cos(e, ref)
    print(f"float32 UNet under bf16 autocast, final-latent cosine: run_generation {c:.6f}  engine {ce:.6f}")
    assert c >= 0.999 and ce >= 0.999
