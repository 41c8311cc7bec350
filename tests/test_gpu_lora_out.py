"""GPU (B200): LoRA on the cross-attention out projection (``attn2.to_out.0``, peft 0.10.0 ``lora.Linear``:
``Y = O Wo^T + bo + s B_o A_o dropout(O)``) in inference and training, against the fp64 oracle with that formula at the
out projection (tests/lora_out_reference.py) and torch autograd through it.  Tolerances are those of test_gpu_kernels.py /
test_gpu_f16.py (forward) and test_gpu_backward.py / test_gpu_train.py (gradients)."""
import pytest
import torch

from oracle import cases, detgen
from oracle.processor_oracle import LoraWeights
from tests.helpers import build_product_layer, force_fusion_seed
from tests.lora_out_reference import clone_with_out_lora_oracle_processors, dual_branch_attention_out_lora

pytestmark = pytest.mark.gpu

F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64
FWD_TOL = {F32: 1e-4, BF16: 2e-2, F16: 2e-2}
REL = {F32: 1e-4, BF16: 4e-2}
FACTORS = ("to_q", "to_k", "to_v", "to_out")
OUT_TARGETS = ("attn2.to_k", "attn2.to_v", "attn2.to_q", "attn2.to_out.0")


def _rel(a, b):
    a, b = a.double(), b.double().to(a.device)
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _out_lora(case, r, dtype=F32):
    """The case's to_out LoRA: non-zero B, scaling 1 so that the low-rank term is of the order of Y at every rank."""
    s = case.seed * 100 + 60
    return LoraWeights(A=detgen.uniform_linear(r, case.C, s, dtype), B=detgen.uniform((case.C, r), s + 1, -0.3, 0.3, dtype),
                       scaling=1.0)


def _weights(case, r_out, dtype=F64, device=None):
    w = cases.proc_weights(case, dtype)
    if r_out:
        w.lora["to_out"] = _out_lora(case, r_out, dtype)
    return w.to(device=device)


def _layer(case, dev, r_out, fresh=False):
    """build_product_layer + a LoRA-wrapped to_out[0] holding the case's factors (``fresh``: peft's init, B = 0)."""
    from photoverse_b200.lora import LoraLinear
    attn, proc = build_product_layer(case, dev)
    if r_out:
        lw = _out_lora(case, r_out)
        wrapped = LoraLinear(attn.to_out[0], r=r_out, lora_alpha=lw.scaling * r_out)
        if not fresh:
            with torch.no_grad():
                wrapped.lora_A["default"].weight.copy_(lw.A)
                wrapped.lora_B["default"].weight.copy_(lw.B)
        attn.to_out[0] = wrapped
    return attn, proc


def _factor(attn, name, which):
    m = attn.to_out[0] if name == "to_out" else getattr(attn, name)
    return getattr(m, "lora_" + which)["default"].weight


def _trainable(attn, proc):
    for p in attn.parameters():
        p.requires_grad_(False)
    out = {"to_k_ip": proc.to_k_ip[0].weight, "to_v_ip": proc.to_v_ip[0].weight}
    for name in FACTORS:
        m = attn.to_out[0] if name == "to_out" else getattr(attn, name)
        if hasattr(m, "lora_A"):
            out[name + ".A"], out[name + ".B"] = _factor(attn, name, "A"), _factor(attn, name, "B")
    for p in out.values():
        p.requires_grad_(True)
    return out


def _oracle_grads(w, x, text, img, gy, gv, wt, wi, drop=None):
    """Autograd through the oracle in the dtype / on the device of ``w`` (fp64 on the GPU)."""
    dev, dt = w.to_q.device, w.to_q.dtype
    leaves = {k: t.to(dev, dt).clone().requires_grad_(True) for k, t in (("x", x), ("text", text), ("img", img))}
    w.to_k_ip.requires_grad_(True)
    w.to_v_ip.requires_grad_(True)
    for lw in w.lora.values():
        lw.A.requires_grad_(True)
        lw.B.requires_grad_(True)
    y, vn = dual_branch_attention_out_lora(leaves["x"], leaves["text"], leaves["img"], w, wt, wi, drop)
    ((y * gy.to(dev, dt)).sum() + (vn.squeeze(-1) * gv.to(dev, dt)).sum()).backward()
    out = {k: v.grad for k, v in leaves.items()}
    out["to_k_ip"], out["to_v_ip"] = w.to_k_ip.grad, w.to_v_ip.grad
    for name, lw in w.lora.items():
        out[name + ".A"], out[name + ".B"] = lw.A.grad, lw.B.grad
    return y.detach(), vn.detach(), out


def _train_call(attn, proc, case, dtype, dev, gy, gv, cuda_seed=None):
    x, text, img = cases.proc_inputs(case, F32)
    xd, td, im = (t.to(dev, dtype).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)          # torch.manual_seed: re-seeds the CUDA generator too
    if cuda_seed is not None:
        torch.cuda.manual_seed(cuda_seed)
    with torch.enable_grad():
        y = attn(xd, encoder_hidden_states=(td, im))
        assert proc.last_fusion == (case.w_text, case.w_img)
        vn = proc.to_v_ip_norm
        ((y.float() * gy.to(dev)).sum() + (vn.float().squeeze(-1) * gv.to(dev)).sum()).backward()
    return y.detach(), vn.detach(), {"x": xd.grad, "text": td.grad, "img": im.grad}


def _check_grads(got, ref, tol):
    assert "to_out.A" in ref and "to_out.B" in ref
    for k, r in ref.items():
        if r is None or r.abs().max() == 0:      # a parameter of a branch the fusion rule dropped
            assert got[k] is None or got[k].abs().max().item() <= 1e-6, k
            continue
        assert got[k] is not None, f"no gradient for {k}"
        e = _rel(got[k], r)
        assert e <= tol, f"{k}: relative error {e:.3e} > {tol}"


# ---- inference ---------------------------------------------------------------------------------------------------
SHAPES = [(2, 4096, 320, 5), (2, 1024, 640, 5), (2, 256, 1280, 5), (2, 64, 1280, 16)]     # the SD-1.5 attn2 layers


@pytest.mark.parametrize("r", [4, 16, 128])
@pytest.mark.parametrize("B,S,C,Li", SHAPES, ids=[f"S{s}_C{c}" for _, s, c, _ in SHAPES])
def test_forward_matches_oracle(cuda_device, B, S, C, Li, r):
    """Merged Wo + s B_o A_o in bf16, fp16 and fp32, both launch forms (the single launch and attention + GEMM)."""
    from photoverse_b200 import _lib
    case = cases.ProcCase(f"out_fwd_{S}_{C}", B=B, S=S, C=C, Li=Li, lora_r=8, seed=120 + r)
    attn, proc = _layer(case, cuda_device, r)
    x, text, img = cases.proc_inputs(case, F32)
    w = _weights(case, r, F64, cuda_device)
    with torch.no_grad():
        args = [t.to(cuda_device, F64) for t in (x, text, img)]
        y_ref, vn_ref = dual_branch_attention_out_lora(*args, w)
        w.lora.pop("to_out")
        y_plain, _ = dual_branch_attention_out_lora(*args, w)
    assert (y_ref - y_plain).abs().max().item() > 0.05                 # the low-rank term is far above the tolerances
    fuses = (2, 0) if S > 128 else (1,)
    for dtype in (BF16, F16, F32):
        for fuse in (fuses if dtype != F32 else (1,)):
            _lib.set_option("fuse_out", fuse)
            try:
                with torch.no_grad():
                    y = attn(x.to(cuda_device, dtype), encoder_hidden_states=(text.to(cuda_device, dtype),
                                                                               img.to(cuda_device, dtype)))
            finally:
                _lib.set_option("fuse_out", 1)
            assert y.dtype == dtype
            err = (y.double() - y_ref).abs().max().item()
            assert err <= FWD_TOL[dtype], f"{dtype} fuse_out={fuse}: max-abs {err}"
            assert (proc.to_v_ip_norm.double().squeeze(-1) / vn_ref.squeeze(-1) - 1).abs().max().item() <= 1e-2


def test_changing_the_out_factors_repacks(cuda_device):
    """An in-place update of B_o (what an optimizer step does) re-packs Wo: the next call follows the new factors."""
    case = cases.ProcCase("out_repack", B=2, S=512, C=640, Li=5, lora_r=8, seed=131)
    attn, proc = _layer(case, cuda_device, 8)
    x, text, img = (t.to(cuda_device, BF16) for t in cases.proc_inputs(case, F32))
    w = _weights(case, 8, F64, cuda_device)
    args = [t.double() for t in (x, text, img)]
    with torch.no_grad():
        y0 = attn(x, encoder_hidden_states=(text, img))
        _factor(attn, "to_out", "B").mul_(-2.0)
        y1 = attn(x, encoder_hidden_states=(text, img))
        w.lora["to_out"].B.mul_(-2.0)
        y_ref, _ = dual_branch_attention_out_lora(*args, w)
    assert (y1.double() - y_ref).abs().max().item() <= 2e-2
    assert (y1.double() - y0.double()).abs().max().item() > 0.1


def test_generation_launches_and_output_with_a_merged_out_lora(cuda_device):
    """The captured UNet evaluation launches the same kernels with and without a to_out LoRA (it is merged into the packed
    Wo), and the engine's latents with one follow the oracle arm (K/V cache and CUDA graphs on)."""
    from oracle.host_reference import clone_adapter_as_oracle
    from photoverse_b200.host.pipeline import GenerationEngine, run_generation, synthetic_inputs
    from photoverse_b200.lora import inject_lora
    from tests.test_gpu_pipeline import _cos, _models
    launches, lat = {}, {}
    for arm, targets in (("qkv", OUT_TARGETS[:3]), ("qkv_out", OUT_TARGETS)):
        unet, ia, ta = _models(cuda_device, BF16)
        inject_lora(unet, r=8, target_modules=targets)
        g = torch.Generator().manual_seed(3)
        with torch.no_grad():
            for n, p in unet.named_parameters():
                if "lora_B" in n:
                    p.copy_(0.05 * torch.randn(p.shape, generator=g))
        inp = synthetic_inputs(2, 32, seed=13, device=cuda_device, dtype=BF16)
        eng = GenerationEngine(unet, ia, ta, batch=2, latent=32, num_steps=10, dtype=BF16, device=cuda_device)
        eng.load_inputs(inp)
        lat[arm] = eng.generate().clone()
        launches[arm] = eng.launches_per_eval
        eng.close()
    ref_unet = clone_with_out_lora_oracle_processors(unet)
    ref_ia, ref_ta = clone_adapter_as_oracle(ia, cuda_device, BF16), clone_adapter_as_oracle(ta, cuda_device, BF16)
    ref = run_generation(ref_unet, ref_ia, ref_ta, inp, num_steps=10, mode="two_call", use_cuda_graph=False, kv_cache=False)
    assert launches["qkv"] == launches["qkv_out"] > 0
    c = _cos(lat["qkv_out"], ref)
    print(f"to_out LoRA generation: final-latent cosine {c:.6f}, launches per UNet evaluation {launches['qkv_out']}")
    assert c >= 0.999


# ---- training: merged path ---------------------------------------------------------------------------------------
BWD_CASES = [
    cases.ProcCase("out_bwd_c320_r4", B=2, S=200, C=320, Li=5, lora_r=4, seed=141),
    cases.ProcCase("out_bwd_c640_r16_textonly", B=1, S=256, C=640, Li=3, lora_r=16, w_text=2.0, w_img=0.0, seed=142),
    cases.ProcCase("out_bwd_c1280_r16", B=2, S=256, C=1280, Li=5, lora_r=16, seed=143),
    cases.ProcCase("out_bwd_c1280_r128_imgonly", B=1, S=64, C=1280, Li=16, lora_r=128, w_text=0.0, w_img=2.0, seed=144),
    cases.ProcCase("out_bwd_c320_r128", B=2, S=600, C=320, Li=5, lora_r=128, seed=145),
]


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", BWD_CASES, ids=lambda c: c.name)
def test_backward_matches_oracle_autograd(cuda_device, case, dtype):
    """Every gradient -- x, text, img, to_k_ip, to_v_ip and the A / B factors of q, k, v and out -- against autograd
    through the oracle in fp64.  Ranks 4 / 16 take the fused pv_lora_bwd, rank 128 the GEMM route."""
    attn, proc = _layer(case, cuda_device, case.lora_r)
    trainable = _trainable(attn, proc)
    g = torch.Generator().manual_seed(case.seed)
    gy, gv = torch.randn(case.B, case.S, case.C, generator=g), torch.randn(case.B, case.H, case.Li, generator=g)
    y, vn, got = _train_call(attn, proc, case, dtype, cuda_device, gy, gv)
    got.update({k: p.grad for k, p in trainable.items()})
    assert all(got[k].dtype == F32 for k in trainable if got[k] is not None)
    x, text, img = cases.proc_inputs(case, F32)
    y_ref, vn_ref, ref = _oracle_grads(_weights(case, case.lora_r, F64, cuda_device), x, text, img, gy, gv,
                                       case.w_text, case.w_img)
    assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[dtype]
    assert got["to_out.A"] is not None and got["to_out.B"] is not None      # the fusion rule never drops to_out
    _check_grads(got, ref, REL[dtype])


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
def test_freshly_injected_out_lora_changes_nothing(cuda_device, dtype):
    """peft initialises B_o = 0: outputs and every gradient the layer had before are bit-identical, in inference and on
    the merged training path."""
    case = cases.ProcCase("out_fresh", B=2, S=300, C=640, Li=5, lora_r=8, seed=151)
    g = torch.Generator().manual_seed(5)
    gy, gv = torch.randn(case.B, case.S, case.C, generator=g), torch.randn(case.B, case.H, case.Li, generator=g)
    runs = {}
    for r_out in (0, 8):
        attn, proc = _layer(case, cuda_device, r_out, fresh=True)
        x, text, img = (t.to(cuda_device, dtype) for t in cases.proc_inputs(case, F32))
        with torch.no_grad():
            y_inf = attn(x, encoder_hidden_states=(text, img))
        trainable = _trainable(attn, proc)
        y, vn, got = _train_call(attn, proc, case, dtype, cuda_device, gy, gv)
        got.update({k: p.grad for k, p in trainable.items()})
        runs[r_out] = (y_inf, y, vn, got)
    a, b = runs[0], runs[8]
    for name, u, v in (("inference y", a[0], b[0]), ("training y", a[1], b[1]), ("to_v_ip_norm", a[2], b[2])):
        assert torch.equal(u, v), name
    for k, t in a[3].items():
        assert torch.equal(t, b[3][k]), k
    assert b[3]["to_out.B"] is not None and b[3]["to_out.B"].abs().max() > 0


# ---- training: LoRA-dropout path ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", [
    cases.ProcCase("out_drop_c320", B=2, S=200, C=320, Li=5, lora_r=8, seed=161),
    cases.ProcCase("out_drop_c640_r4_textonly", B=1, S=256, C=640, Li=1, lora_r=4, w_text=2.0, w_img=0.0, seed=162),
    cases.ProcCase("out_drop_c1280_r16", B=1, S=64, C=1280, Li=3, lora_r=16, seed=163),
], ids=lambda c: c.name)
def test_lora_dropout_matches_oracle(cuda_device, case, dtype):
    """p = 0.1 on all four projections: forward and every gradient against the oracle with the same keep-masks, re-drawn
    with ``torch.native_dropout`` from the same CUDA generator state in the reference's order q, k, v, out."""
    p_drop = 0.1
    attn, proc = _layer(case, cuda_device, case.lora_r)
    for name in ("to_q", "to_k", "to_v"):
        getattr(attn, name).lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.to_out[0].lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.train()
    trainable = _trainable(attn, proc)
    assert proc.lora_dropout_active(attn)
    g = torch.Generator().manual_seed(case.seed)
    gy, gv = torch.randn(case.B, case.S, case.C, generator=g), torch.randn(case.B, case.H, case.Li, generator=g)
    y, vn, got = _train_call(attn, proc, case, dtype, cuda_device, gy, gv, cuda_seed=1000 + case.seed)
    got.update({k: p.grad for k, p in trainable.items()})
    x, text, img = cases.proc_inputs(case, F32)
    torch.cuda.manual_seed(1000 + case.seed)
    drop = {}
    for name, shape in (("to_q", x.shape), ("to_k", text.shape), ("to_v", text.shape), ("to_out", x.shape)):
        _, mask = torch.native_dropout(torch.zeros(shape, device=cuda_device, dtype=dtype), p_drop, True)
        drop[name] = (mask.to(cuda_device), p_drop)
    assert not torch.equal(drop["to_out"][0], drop["to_q"][0])
    w = _weights(case, case.lora_r, F64, cuda_device)
    y_ref, vn_ref, ref = _oracle_grads(w, x, text, img, gy, gv, case.w_text, case.w_img, drop)
    assert (y.double() - y_ref).abs().max().item() <= FWD_TOL[dtype]
    only_qkv = dict(drop)
    only_qkv.pop("to_out")
    with torch.no_grad():
        y_nout, _ = dual_branch_attention_out_lora(*(t.to(cuda_device, F64) for t in (x, text, img)),
                                          _weights(case, case.lora_r, F64, cuda_device), case.w_text, case.w_img, only_qkv)
    assert (y_nout - y_ref).abs().max().item() > 1e-2                  # the out-projection mask matters
    _check_grads(got, ref, REL[dtype])


# ---- a pending backward keeps its forward's weights --------------------------------------------------------------
@pytest.mark.parametrize("p_drop", [0.0, 0.1], ids=["merged", "lora_dropout"])
def test_backward_uses_the_weights_its_forward_ran_with(cuda_device, p_drop):
    """With a to_out LoRA the packed Wo is re-packed whenever its sources change.  The frozen base Wo -- part of that pack
    but not of the saved tensors -- changed in place between a training forward and its backward (with a call in between
    that re-packs) must leave the pending backward's gradients, the to_out factors' included, equal to a fresh layer's.
    The LoRA factors are saved tensors: changing one in place makes the backward raise, as torch autograd does."""
    case = cases.ProcCase("out_pending", B=2, S=200, C=320, Li=5, lora_r=8, seed=171)

    def run(change):
        attn, proc = _layer(case, cuda_device, 8)
        if p_drop:
            for m in (attn.to_q, attn.to_k, attn.to_v, attn.to_out[0]):
                m.lora_dropout["default"] = torch.nn.Dropout(p_drop)
            attn.train()
        trainable = _trainable(attn, proc)
        x, text, img = (t.to(cuda_device, BF16).requires_grad_(True) for t in cases.proc_inputs(case, F32))
        force_fusion_seed(1.0, 1.0)
        torch.cuda.manual_seed(1000 + case.seed)
        with torch.enable_grad():
            y = attn(x, encoder_hidden_states=(text, img))
            loss = y.float().square().sum() + proc.to_v_ip_norm.float().sum()
            if change:
                with torch.no_grad():
                    if change == "base":
                        attn.to_out[0].base_layer.weight.mul_(-2.0)
                    else:
                        _factor(attn, "to_out", "B").mul_(-2.0)
                attn(x, encoder_hidden_states=(text, img))
        loss.backward()
        return [y.detach(), x.grad, text.grad, img.grad] + [p.grad for p in trainable.values()]

    fresh, changed = run(None), run("base")
    for i, (a, b) in enumerate(zip(fresh, changed)):
        assert torch.equal(a, b), i
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        run("factor")


# ---- Trainer --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arm", ["bf16", "f32_autocast"])
def test_trainer_step_with_out_lora(cuda_device, arm):
    """A training step of a reduced SD-1.5 UNet with LoRA on q / k / v / out: a bf16 backbone with float32 masters of the
    trainable set (bench.py's training configuration), and a float32 model under bf16 autocast.  Loss and gradients
    against the fp32 oracle arm at test_gpu_train.py's bf16 tolerance; the to_out factors get float32 gradients and move."""
    import photoverse_b200 as pv
    from oracle import adapter_oracle
    from photoverse_b200.host.parallel import trainable_named_parameters
    from photoverse_b200.host.train_step import Trainer, synthetic_train_batch
    from photoverse_b200.host.unet_sd15 import UNetSD15
    from photoverse_b200.lora import inject_lora
    from photoverse_b200.unet import get_visual_cross_attention_values_norm
    torch.manual_seed(0)
    unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
    ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
    unet.requires_grad_(False)
    inject_lora(unet, r=8, target_modules=OUT_TARGETS)
    g = torch.Generator().manual_seed(1)
    for n, p in unet.named_parameters():
        if "to_k_ip" in n or "to_v_ip" in n:
            p.requires_grad_(True)
        if "lora_B" in n:
            with torch.no_grad():
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
    for m in (unet, ia, ta):
        m.to(device=cuda_device, dtype=F32)
    if arm == "bf16":
        unet.to(BF16)
        for n, p in unet.named_parameters():
            if p.requires_grad:
                p.data = p.data.float()
    unet.eval()
    data_dt, ac = (BF16, None) if arm == "bf16" else (F32, BF16)
    ref_unet = clone_with_out_lora_oracle_processors(unet).float()
    b = synthetic_train_batch(2, latent=16, seed=3, device=cuda_device, dtype=data_dt)
    tr = Trainer(unet, ia, ta, lr=1e-3, autocast_dtype=ac)
    named = trainable_named_parameters(unet, ia, ta)
    out_names = [n for n, _ in named if "to_out.0.lora_" in n]
    assert len(out_names) == 8
    torch.manual_seed(0)
    with torch.enable_grad(), torch.autocast("cuda", dtype=BF16, enabled=ac is not None, cache_enabled=False):
        loss, _ = tr.loss(b)
    loss.backward()
    got = {n: p.grad.detach().clone() for n, p in named if p.grad is not None}
    r16 = lambda t: t.to(BF16).float()
    torch.manual_seed(0)
    with torch.enable_grad():
        emb = [r16(e) for e in b.clip_hidden]
        concept = adapter_oracle.adapter_forward(emb, dict(ta.named_parameters()), None)
        img_tokens = adapter_oracle.adapter_forward(emb, dict(ia.named_parameters()), None)
        pred = ref_unet(r16(b.noisy_latents), b.timesteps.float(), encoder_hidden_states=(r16(b.text), img_tokens)).sample
        l_vis = get_visual_cross_attention_values_norm(ref_unet).mean()
        ref_loss = torch.nn.functional.mse_loss(pred, b.noise.float()) + 0.01 * concept.abs().mean() + 0.001 * l_vis
    for m in (ia, ta):
        for p in m.parameters():
            p.grad = None
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 3e-2 * abs(ref_loss.item())
    ref_named = trainable_named_parameters(ref_unet, ia, ta)
    checked = 0
    for (n, p), (n_ref, p_ref) in zip(named, ref_named):
        assert n == n_ref
        if p_ref.grad is None or p_ref.grad.abs().max() == 0:
            assert n not in got or got[n].abs().max().item() <= 1e-6, n
            continue
        e = _rel(got[n].float(), p_ref.grad.float())
        assert e <= 1.0e-1, f"{n}: relative error {e:.3e}"
        checked += 1
    assert checked > 100 and all(n in got for n in out_names)
    before = {n: p.detach().clone() for n, p in named}
    torch.manual_seed(0)
    loss, _ = tr.step(b)
    assert torch.isfinite(loss)
    params = dict(named)
    for n in out_names:
        p = params[n]
        assert p.dtype == F32 and p.grad is not None and p.grad.dtype == F32, n
        assert not torch.equal(p, before[n]), n
