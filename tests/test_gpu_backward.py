"""GPU (B200): the training path -- forward AND backward in the CUDA library through the C ABI -- against
``torch.autograd`` through the CPU oracle (which follows the reference line by line, oracle/processor_oracle.py).

Metric: relative Frobenius error ||g - g_ref|| / ||g_ref|| per gradient tensor -- fp32 mode <= 1e-4, bf16 mode <= 4e-2
(processor) / 6e-2 (adapter: bf16 weights and activations through two LayerNorm+LeakyReLU layers, where a pre-activation
within bf16 noise of zero flips the LeakyReLU slope of that single element; with the 2-3 rows of the CLS branch in these
small cases such a flip moves one entry by its own magnitude, so a max-abs metric would test luck, not arithmetic)."""
import pytest
import torch

from oracle import adapter_oracle, cases
from oracle.processor_oracle import dual_branch_attention
from tests.helpers import build_product_layer, force_fusion_seed

pytestmark = pytest.mark.gpu

REL = {torch.float32: 1e-4, torch.bfloat16: 4e-2}


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _oracle_grads(case, x, text, img, gy, gv, wt, wi, drop=None):
    w = cases.proc_weights(case, torch.float64)
    leaves = {"x": x.double().clone().requires_grad_(True), "text": text.double().clone().requires_grad_(True),
              "img": img.double().clone().requires_grad_(True)}
    w.to_k_ip.requires_grad_(True)
    w.to_v_ip.requires_grad_(True)
    for lw in w.lora.values():
        lw.A.requires_grad_(True)
        lw.B.requires_grad_(True)
    y, vn = dual_branch_attention(leaves["x"], leaves["text"], leaves["img"], w, wt, wi, drop)
    loss = (y * gy.double()).sum() + (vn.squeeze(-1) * gv.double()).sum()
    loss.backward()
    out = {k: v.grad for k, v in leaves.items()}
    out["to_k_ip"], out["to_v_ip"] = w.to_k_ip.grad, w.to_v_ip.grad
    for name, lw in w.lora.items():
        out[name + ".A"], out[name + ".B"] = lw.A.grad, lw.B.grad
    return y.detach(), vn.detach(), out


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", [
    cases.ProcCase("bwd_c320", B=2, S=200, C=320, Li=5, lora_r=8, seed=71),
    cases.ProcCase("bwd_c640_textonly", B=1, S=128, C=640, Li=1, lora_r=4, w_text=2.0, w_img=0.0, seed=72),
    cases.ProcCase("bwd_c1280_imgonly", B=1, S=64, C=1280, Li=16, w_text=0.0, w_img=2.0, seed=73),
    cases.ProcCase("bwd_c320_long", B=2, S=600, C=320, Li=4, seed=74),
], ids=lambda c: c.name)
def test_processor_backward_matches_oracle_autograd(cuda_device, case, dtype):
    attn, proc = build_product_layer(case, cuda_device)
    for p in attn.parameters():
        p.requires_grad_(False)
    trainable = {"to_k_ip": proc.to_k_ip[0].weight, "to_v_ip": proc.to_v_ip[0].weight}
    for name in ("to_q", "to_k", "to_v"):
        m = getattr(attn, name)
        if hasattr(m, "lora_A"):
            trainable[name + ".A"] = m.lora_A["default"].weight
            trainable[name + ".B"] = m.lora_B["default"].weight
    for p in trainable.values():
        p.requires_grad_(True)
    x, text, img = cases.proc_inputs(case, torch.float32)
    g = torch.Generator().manual_seed(case.seed)
    gy = torch.randn(case.B, case.S, case.C, generator=g)
    gv = torch.randn(case.B, case.H, case.Li, generator=g)
    xd, td, im = (t.to(cuda_device, dtype).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)
    with torch.enable_grad():
        y = attn(xd, encoder_hidden_states=(td, im))
        assert proc.last_fusion == (case.w_text, case.w_img)
        vn = proc.to_v_ip_norm
        loss = (y.float() * gy.to(cuda_device)).sum() + (vn.float().squeeze(-1) * gv.to(cuda_device)).sum()
    loss.backward()
    y_ref, vn_ref, ref = _oracle_grads(case, x, text, img, gy, gv, case.w_text, case.w_img)
    assert (y.detach().float().cpu() - y_ref.float()).abs().max().item() <= (1e-4 if dtype == torch.float32 else 2e-2)
    got = {"x": xd.grad, "text": td.grad, "img": im.grad}
    got.update({k: p.grad for k, p in trainable.items()})
    for k, r in ref.items():
        if r is None or r.abs().max() == 0:   # e.g. image-branch parameters when the fusion rule dropped that branch
            assert got[k] is None or got[k].abs().max().item() <= 1e-6
            continue
        assert got[k] is not None, f"no gradient for {k}"
        e = _rel(got[k], r)
        assert e <= REL[dtype], f"{k}: relative error {e:.3e} > {REL[dtype]}"


def _oracle_grads_on(device, dtype, case, x, text, img, gy, gv, wt, wi):
    """The same checker evaluated on ``device`` in ``dtype`` (fp32 on the GPU for the full-size shapes, where the CPU
    fp64 run would take minutes)."""
    w = cases.proc_weights(case, dtype).to(device=device)
    leaves = {k: t.to(device, dtype).clone().requires_grad_(True) for k, t in (("x", x), ("text", text), ("img", img))}
    w.to_k_ip.requires_grad_(True)
    w.to_v_ip.requires_grad_(True)
    for lw in w.lora.values():
        lw.A.requires_grad_(True)
        lw.B.requires_grad_(True)
    y, vn = dual_branch_attention(leaves["x"], leaves["text"], leaves["img"], w, wt, wi, None)
    ((y * gy.to(device, dtype)).sum() + (vn.squeeze(-1) * gv.to(device, dtype)).sum()).backward()
    out = {k: v.grad for k, v in leaves.items()}
    out["to_k_ip"], out["to_v_ip"] = w.to_k_ip.grad, w.to_v_ip.grad
    for name, lw in w.lora.items():
        out[name + ".A"], out[name + ".B"] = lw.A.grad, lw.B.grad
    return y.detach(), vn.detach(), out


@pytest.mark.parametrize("case", [
    cases.ProcCase("bwd_full_c320", B=16, S=4096, C=320, Li=5, lora_r=8, seed=91),          # BASELINE config[3] layer shapes:
    cases.ProcCase("bwd_full_c640", B=16, S=1024, C=640, Li=5, lora_r=8, seed=92),          # batch 16 per GPU, latent 64^2
    cases.ProcCase("bwd_full_c1280", B=16, S=256, C=1280, Li=5, lora_r=8, seed=93),
    cases.ProcCase("bwd_full_mid", B=16, S=64, C=1280, Li=5, lora_r=8, seed=94),
    cases.ProcCase("bwd_r128_c320", B=4, S=4096, C=320, Li=5, lora_r=128, seed=95),         # the shipped recipe's LoRA rank
    cases.ProcCase("bwd_r128_c1280_textonly", B=4, S=256, C=1280, Li=5, lora_r=128, w_text=2.0, w_img=0.0, seed=96),
    cases.ProcCase("bwd_r128_c640_imgonly", B=4, S=1024, C=640, Li=5, lora_r=128, w_text=0.0, w_img=2.0, seed=97),
], ids=lambda c: c.name)
def test_processor_backward_full_size_bf16(cuda_device, case):
    """Forward + every gradient at the REAL training shapes (config[3]: B = 16 per GPU, the four attn2 layer shapes at
    latent 64^2; LoRA rank 8 and the shipped recipe's rank 128, prepare_dataset_and_train.sh:2) in bf16, against autograd
    through the oracle evaluated in fp32 on the GPU."""
    dtype = torch.bfloat16
    attn, proc = build_product_layer(case, cuda_device)
    for p in attn.parameters():
        p.requires_grad_(False)
    trainable = {"to_k_ip": proc.to_k_ip[0].weight, "to_v_ip": proc.to_v_ip[0].weight}
    for name in ("to_q", "to_k", "to_v"):
        m = getattr(attn, name)
        trainable[name + ".A"] = m.lora_A["default"].weight
        trainable[name + ".B"] = m.lora_B["default"].weight
    for p in trainable.values():
        p.requires_grad_(True)
    x, text, img = cases.proc_inputs(case, torch.float32)
    g = torch.Generator().manual_seed(case.seed)
    gy = torch.randn(case.B, case.S, case.C, generator=g)
    gv = torch.randn(case.B, case.H, case.Li, generator=g)
    xd, td, im = (t.to(cuda_device, dtype).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)
    with torch.enable_grad():
        y = attn(xd, encoder_hidden_states=(td, im))
        assert proc.last_fusion == (case.w_text, case.w_img)
        vn = proc.to_v_ip_norm
        loss = (y.float() * gy.to(cuda_device)).sum() + (vn.float().squeeze(-1) * gv.to(cuda_device)).sum()
    loss.backward()
    y_ref, vn_ref, ref = _oracle_grads_on(cuda_device, torch.float32, case, x, text, img, gy, gv, case.w_text, case.w_img)
    assert (y.detach().float() - y_ref).abs().max().item() <= 2e-2
    assert _rel(vn.float().squeeze(-1), vn_ref.squeeze(-1)) <= 1e-2
    got = {"x": xd.grad, "text": td.grad, "img": im.grad}
    got.update({k: p.grad for k, p in trainable.items()})
    for k, r in ref.items():
        if r is None or r.abs().max() == 0:
            assert got[k] is None or got[k].abs().max().item() <= 1e-6, k
            continue
        assert got[k] is not None, f"no gradient for {k}"
        e = _rel(got[k], r)
        assert e <= REL[dtype], f"{k}: relative error {e:.3e} > {REL[dtype]}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("case", [
    cases.ProcCase("drop_c320", B=2, S=200, C=320, Li=5, lora_r=8, seed=76),
    cases.ProcCase("drop_c640_r4_textonly", B=1, S=256, C=640, Li=1, lora_r=4, w_text=2.0, w_img=0.0, seed=77),
    cases.ProcCase("drop_c1280", B=1, S=64, C=1280, Li=3, lora_r=16, seed=78),
], ids=lambda c: c.name)
def test_processor_lora_dropout_training_matches_oracle(cuda_device, case, dtype):
    """LoRA dropout p = 0.1 in training mode (the reference default, train.py:264-269): forward and every gradient vs
    the oracle evaluated with the SAME keep-masks.  The masks are re-drawn here with ``torch.native_dropout`` from the
    same CUDA generator state in the reference's call order (to_q, to_k, to_v), which also pins the RNG contract."""
    p_drop = 0.1
    attn, proc = build_product_layer(case, cuda_device)
    for name in ("to_q", "to_k", "to_v"):
        getattr(attn, name).lora_dropout["default"] = torch.nn.Dropout(p_drop)
    attn.train()
    for p in attn.parameters():
        p.requires_grad_(False)
    trainable = {"to_k_ip": proc.to_k_ip[0].weight, "to_v_ip": proc.to_v_ip[0].weight}
    for name in ("to_q", "to_k", "to_v"):
        m = getattr(attn, name)
        trainable[name + ".A"] = m.lora_A["default"].weight
        trainable[name + ".B"] = m.lora_B["default"].weight
    for p in trainable.values():
        p.requires_grad_(True)
    assert proc.lora_dropout_active(attn)
    x, text, img = cases.proc_inputs(case, torch.float32)
    g = torch.Generator().manual_seed(case.seed)
    gy = torch.randn(case.B, case.S, case.C, generator=g)
    gv = torch.randn(case.B, case.H, case.Li, generator=g)
    xd, td, im = (t.to(cuda_device, dtype).requires_grad_(True) for t in (x, text, img))
    force_fusion_seed(case.w_text, case.w_img)
    torch.cuda.manual_seed(1000 + case.seed)
    with torch.enable_grad():
        y = attn(xd, encoder_hidden_states=(td, im))
        vn = proc.to_v_ip_norm
        loss = (y.float() * gy.to(cuda_device)).sum() + (vn.float().squeeze(-1) * gv.to(cuda_device)).sum()
    loss.backward()
    # the reference's draws: nn.Dropout on to_q's input, then to_k's, then to_v's
    torch.cuda.manual_seed(1000 + case.seed)
    drop = {}
    for name, t in (("to_q", xd), ("to_k", td), ("to_v", td)):
        _, mask = torch.native_dropout(t.detach(), p_drop, True)
        drop[name] = (mask.cpu(), p_drop)
    assert not torch.equal(drop["to_k"][0], drop["to_v"][0])
    y_ref, vn_ref, ref = _oracle_grads(case, x, text, img, gy, gv, case.w_text, case.w_img, drop)
    assert (y.detach().float().cpu() - y_ref.float()).abs().max().item() <= (1e-4 if dtype == torch.float32 else 2e-2)
    # and the masks matter: the no-dropout oracle is measurably different
    y_nodrop, _, _ = _oracle_grads(case, x, text, img, gy, gv, case.w_text, case.w_img, None)
    assert (y_nodrop - y_ref).abs().max().item() > 1e-3
    got = {"x": xd.grad, "text": td.grad, "img": im.grad}
    got.update({k: p.grad for k, p in trainable.items()})
    for k, r in ref.items():
        if r is None or r.abs().max() == 0:
            assert got[k] is None or got[k].abs().max().item() <= 1e-6
            continue
        assert got[k] is not None, f"no gradient for {k}"
        e = _rel(got[k], r)
        assert e <= REL[dtype], f"{k}: relative error {e:.3e} > {REL[dtype]}"
    # eval mode: dropout is the identity and the merged-weight fast path is taken again
    attn.eval()
    assert not proc.lora_dropout_active(attn)
    with torch.no_grad():
        y_eval = attn(xd.detach(), encoder_hidden_states=(td.detach(), im.detach()))
    w = cases.proc_weights(case, torch.float64)
    y_eval_ref, _ = dual_branch_attention(x.double(), text.double(), img.double(), w, 1.0, 1.0)
    assert (y_eval.float().cpu() - y_eval_ref.float()).abs().max().item() <= (1e-4 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("B,T,token_index", [(2, 2, None), (3, 3, 1)])
def test_adapter_backward_matches_oracle_autograd(cuda_device, dtype, B, T, token_index):
    from photoverse_b200 import PhotoVerseAdapter
    sd = adapter_oracle.make_state_dict(T, 90 + T)
    ad = PhotoVerseAdapter(num_tokens=T)
    ad.load_state_dict(sd, strict=True)
    ad.to(cuda_device)
    case = cases.AdapterCase("bwd", B=B, T=T, token_index=token_index, seed=91)
    embs = cases.adapter_inputs(case)
    g = torch.Generator().manual_seed(5)
    n_out = T if token_index is None else 1
    gy = torch.randn(B, n_out, 768, generator=g)
    with torch.enable_grad():
        y = ad([e.to(cuda_device, dtype) for e in embs], token_index=token_index)
        (y.float() * gy.to(cuda_device)).sum().backward()
    sd64 = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    y_ref = adapter_oracle.adapter_forward([e.double() for e in embs], sd64, token_index)
    (y_ref * gy.double()).sum().backward()
    assert (y.detach().float().cpu() - y_ref.detach().float()).abs().max().item() <= (1e-4 if dtype == torch.float32 else 4e-2)
    used = range(T) if token_index is None else [token_index]
    checked = 0
    for name, p in ad.named_parameters():
        head = int(name.split(".")[0].split("_")[-1])
        if head not in used:
            assert p.grad is None or p.grad.abs().max().item() == 0
            continue
        r = sd64[name].grad
        e = _rel(p.grad, r)
        # LeakyReLU kinks: a pre-activation within rounding noise of zero (fp32: ~1e-6 of 5e5 patch pre-activations per
        # layer -> O(1) expected flips; bf16: ~1 %) flips that element's slope, which perturbs the whole weight gradient
        # by a rank-1 term of relative Frobenius size ~1/sqrt(rows*1024) per flip (~1e-3 here).  Arithmetic errors
        # proper are < 1e-5 (fp32): the processor test above, which has no kinks, holds 1e-4.
        tol = 5e-3 if dtype == torch.float32 else 1e-1
        assert e <= tol, f"{name}: relative error {e:.3e} > {tol}"
        checked += 1
    assert checked == 20 * len(list(used))


def test_backward_is_deterministic(cuda_device):
    case = cases.ProcCase("det", B=2, S=512, C=320, Li=5, lora_r=8, seed=75)
    outs = []
    for _ in range(2):
        attn, proc = build_product_layer(case, cuda_device)
        for n, p in attn.named_parameters():
            p.requires_grad_("lora_" in n or "to_k_ip" in n or "to_v_ip" in n)
        x, text, img = (t.to(cuda_device, torch.bfloat16) for t in cases.proc_inputs(case, torch.float32))
        x.requires_grad_(True)
        force_fusion_seed(1.0, 1.0)
        with torch.enable_grad():
            y = attn(x, encoder_hidden_states=(text, img))
            (y.float().square().sum() + proc.to_v_ip_norm.float().sum()).backward()
        outs.append((x.grad.clone(), proc.to_k_ip[0].weight.grad.clone(), attn.to_q.lora_A["default"].weight.grad.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("p_drop", [0.0, 0.1], ids=["merged", "lora_dropout"])
def test_backward_uses_the_weights_its_forward_ran_with(cuda_device, p_drop):
    """A parameter changed in place between a training forward and its backward -- here to_k_ip, which is part of the
    packed weights but not of the saved tensors -- re-packs the layer on the next call.  The pending backward must keep
    the packed weights (and their transposed copies) of its own forward: its input gradients equal a fresh layer's."""
    case = cases.ProcCase("repack", B=2, S=200, C=320, Li=5, lora_r=8, seed=85)

    def run(change_between):
        attn, proc = build_product_layer(case, cuda_device)
        if p_drop:
            for name in ("to_q", "to_k", "to_v"):
                getattr(attn, name).lora_dropout["default"] = torch.nn.Dropout(p_drop)
            attn.train()
        for n, p in attn.named_parameters():
            p.requires_grad_("lora_" in n or "to_k_ip" in n or "to_v_ip" in n)
        assert proc.lora_dropout_active(attn) == (p_drop > 0)
        x, text, img = (t.to(cuda_device, torch.bfloat16).requires_grad_(True)
                        for t in cases.proc_inputs(case, torch.float32))
        force_fusion_seed(1.0, 1.0)
        torch.cuda.manual_seed(1000 + case.seed)
        with torch.enable_grad():
            y = attn(x, encoder_hidden_states=(text, img))
            loss = y.float().square().sum() + proc.to_v_ip_norm.float().sum()
            if change_between:
                with torch.no_grad():
                    proc.to_k_ip[0].weight.mul_(-2.0)
                attn(x, encoder_hidden_states=(text, img))
        loss.backward()
        return y.detach(), x.grad, text.grad, img.grad

    fresh, changed = run(False), run(True)
    for name, a, b in zip(("y", "x", "text", "img"), fresh, changed):
        assert torch.equal(a, b), name


def test_tensor_core_backward_agrees_with_simt_backward(cuda_device):
    """bf16 training path: the mma.sync attention backward (pv_bwd_mma.cu, default) and the fp32-accumulating SIMT kernel
    (pv_set_option('bwd_mma', 0)) on identical inputs -- two independent implementations of reference :317-420's
    derivative must agree to bf16 rounding."""
    from photoverse_b200 import _lib
    case = cases.ProcCase("mma_vs_simt", B=2, S=300, C=640, Li=5, lora_r=8, seed=79)
    grads = {}
    for flag in (1, 0):
        _lib.set_option("bwd_mma", flag)
        try:
            attn, proc = build_product_layer(case, cuda_device)
            for n, p in attn.named_parameters():
                p.requires_grad_("lora_" in n or "to_k_ip" in n or "to_v_ip" in n)
            x, text, img = (t.to(cuda_device, torch.bfloat16) for t in cases.proc_inputs(case, torch.float32))
            x.requires_grad_(True)
            text.requires_grad_(True)
            force_fusion_seed(1.0, 1.0)
            with torch.enable_grad():
                y = attn(x, encoder_hidden_states=(text, img))
                (y.float().square().sum() + proc.to_v_ip_norm.float().sum()).backward()
            grads[flag] = {"x": x.grad.clone(), "text": text.grad.clone(), "kip": proc.to_k_ip[0].weight.grad.clone(),
                           "vip": proc.to_v_ip[0].weight.grad.clone(), "qA": attn.to_q.lora_A["default"].weight.grad.clone(),
                           "kB": attn.to_k.lora_B["default"].weight.grad.clone()}
        finally:
            _lib.set_option("bwd_mma", 1)
    for k in grads[1]:
        e = _rel(grads[1][k], grads[0][k])
        assert e <= 2e-2, f"{k}: tensor-core vs SIMT backward relative difference {e:.3e}"


@pytest.mark.parametrize("case", [
    cases.ProcCase("tc_c320_ragged", B=2, S=700, C=320, Li=5, lora_r=8, seed=81),          # 77 text keys: compile-time segments
    cases.ProcCase("tc_c640_lt60", B=2, S=384, C=640, Li=3, Lt=60, lora_r=4, seed=82),       # other text lengths: generic path
    cases.ProcCase("tc_c320_li16", B=1, S=2304, C=320, Li=16, seed=83),                      # 9 tiles -> two CTAs per (b, h)
], ids=lambda c: c.name)
def test_tcgen05_backward_agrees_with_the_other_backward_kernels(cuda_device, case):
    """bf16 training path: the tcgen05 attention backward (pv_bwd_tc.cu, default for head_dim 40 / 80), the mma.sync
    kernel (pv_set_option('bwd_tc', 0)) and the fp32-accumulating SIMT kernel ('bwd_mma', 0) -- three independent
    implementations of the derivative of reference :317-420 -- on identical inputs."""
    from photoverse_b200 import _lib
    grads = {}
    for name, opts in (("tc", {"bwd_tc": 1, "bwd_mma": 1}), ("mma", {"bwd_tc": 0, "bwd_mma": 1}), ("simt", {"bwd_tc": 0, "bwd_mma": 0})):
        for k, v in opts.items():
            _lib.set_option(k, v)
        try:
            attn, proc = build_product_layer(case, cuda_device)
            for n, p in attn.named_parameters():
                p.requires_grad_("lora_" in n or "to_k_ip" in n or "to_v_ip" in n)
            x, text, img = (t.to(cuda_device, torch.bfloat16) for t in cases.proc_inputs(case, torch.float32))
            x.requires_grad_(True)
            text.requires_grad_(True)
            img.requires_grad_(True)
            force_fusion_seed(1.0, 1.0)
            with torch.enable_grad():
                y = attn(x, encoder_hidden_states=(text, img))
                (y.float().square().sum() + proc.to_v_ip_norm.float().sum()).backward()
            grads[name] = {"x": x.grad.clone(), "text": text.grad.clone(), "img": img.grad.clone(),
                           "kip": proc.to_k_ip[0].weight.grad.clone(), "vip": proc.to_v_ip[0].weight.grad.clone()}
        finally:
            _lib.set_option("bwd_tc", 1)
            _lib.set_option("bwd_mma", 1)
    for other in ("mma", "simt"):
        for k in grads["tc"]:
            e = _rel(grads["tc"][k], grads[other][k])
            assert e <= 2e-2, f"{k}: tcgen05 vs {other} backward relative difference {e:.3e}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("M,in_f,out_f,r", [(4096 + 7, 320, 320, 8), (1232, 768, 640, 8), (300, 1280, 1280, 4), (2048, 768, 1280, 16),
                                            (65536, 320, 320, 8), (64, 640, 640, 1)])
def test_lora_factor_gradients_fused_kernel(cuda_device, dtype, M, in_f, out_f, r):
    """pv_lora_bwd: dA = s (G B)^T X and dB = s G^T (X A^T) of y = W x + s B (A x) (peft 0.10.0 lora.Linear) in one pass,
    vs autograd through that formula in fp64; G is a strided column slice like the K / V halves of dkv_text."""
    from photoverse_b200 import ops
    g = torch.Generator().manual_seed(M + r)
    x = torch.randn(M, in_f, generator=g).to(cuda_device, dtype)
    gfull = torch.randn(M, 2 * out_f, generator=g).to(cuda_device, dtype)
    gy = gfull[:, out_f:]                                     # row stride 2 * out
    A = (torch.randn(r, in_f, generator=g) / in_f ** 0.5).to(cuda_device)
    Bm = (torch.randn(out_f, r, generator=g) * 0.1).to(cuda_device)
    s_ = 0.25
    out = ops.lora_bwd(x, gy, A, Bm, s_)
    assert out is not None
    dA, dB = out
    Ad, Bd = A.double().requires_grad_(True), Bm.double().requires_grad_(True)
    y = s_ * (x.double() @ Ad.t()) @ Bd.t()
    (y * gy.double()).sum().backward()
    # fp32: FFMA path.  bf16: tensor-core path, the intermediate X A^T / G B (and A, B) rounded to bf16 like the activations
    tol = 1e-4 if dtype == torch.float32 else 1e-2
    assert _rel(dA, Ad.grad) <= tol and _rel(dB, Bd.grad) <= tol
    out2 = ops.lora_bwd(x, gy, A, Bm, s_)
    assert torch.equal(out2[0], dA) and torch.equal(out2[1], dB)          # deterministic
    assert ops.lora_bwd(x[:64], gy[:64], torch.zeros(128, in_f, device=cuda_device), torch.zeros(out_f, 128, device=cuda_device), 1.0) is None
