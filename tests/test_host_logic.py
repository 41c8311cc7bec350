"""CPU: host-side logic that mirrors the reference interface (constructor validation, names, installation,
fusion-rule RNG consumption, LoRA injection, DDIM schedule)."""
import pytest
import torch

import photoverse_b200 as pv
from oracle import adapter_oracle, ref_loader
from photoverse_b200.host.ddim import make_ddim_schedule
from photoverse_b200.host.unet_sd15 import UNetSD15
from photoverse_b200.lora import LoraLinear, inject_lora, linear_parts

SD15_ATTN2 = (["down_blocks.%d.attentions.%d" % (i, j) for i in range(3) for j in range(2)]
              + ["mid_block.attentions.0"] + ["up_blocks.%d.attentions.%d" % (i, j) for i in (1, 2, 3) for j in range(3)])


def test_ctor_validation_matches_reference():
    # attention_processor.py:37-48
    with pytest.raises(ValueError, match="tuple of two floats"):
        pv.PhotoVerseAttnProcessor2_0(320, 768, fusion_rules=[1 / 3, 2 / 3])
    with pytest.raises(ValueError, match="tuple of two floats"):
        pv.PhotoVerseAttnProcessor2_0(320, 768, fusion_rules=(1, 0))
    with pytest.raises(ValueError, match="equal to 1"):
        pv.PhotoVerseAttnProcessor2_0(320, 768, fusion_rules=(0.5, 0.6))
    with pytest.raises(ValueError, match="same length"):
        pv.PhotoVerseAttnProcessor2_0(320, 768, num_tokens=(5,), scale=[1.0, 2.0])
    p = pv.PhotoVerseAttnProcessor2_0(hidden_size=640, cross_attention_dim=768, num_tokens=5)
    assert p.num_tokens == [5] and p.scale == [2.0] and p.to_v_ip_norm is None
    assert sorted(p.state_dict().keys()) == ["to_k_ip.0.weight", "to_v_ip.0.weight"]
    assert p.to_k_ip[0].weight.shape == (640, 768) and p.to_k_ip[0].bias is None


def test_processor_state_dict_and_ctor_match_live_reference():
    """State-dict layout, constructor defaults and ValueError texts against the record in tests/golden/class_layout.json
    and, when PHOTOVERSE_REFERENCE_ROOT names an upstream checkout, against the live upstream classes.  The record's
    `provenance` says where it came from: oracle/make_golden.py rewrites it from the upstream classes; until then it
    holds values recorded from photoverse_b200 itself and pins them against change."""
    import json
    from oracle.make_golden import class_layout
    from tests.helpers import GOLDEN_DIR
    ours = class_layout(pv.PhotoVerseAttnProcessor2_0, pv.PhotoVerseAdapter)
    with open(f"{GOLDEN_DIR}/class_layout.json") as f:
        assert ours == json.load(f)["layout"]
    assert None not in ours["processor_ctor_errors"]
    if ref_loader.reference_available():
        ref = class_layout(ref_loader.load_reference_processor_module().PhotoVerseAttnProcessor2_0,
                           ref_loader.load_reference_adapter_module().PhotoVerseAdapter)
        assert ours == json.loads(json.dumps(ref))


def test_adapter_state_dict_names_match_reference_layout():
    ad = pv.PhotoVerseAdapter(num_tokens=3)
    want = adapter_oracle.make_state_dict(3, 1)
    assert {k: tuple(v.shape) for k, v in ad.state_dict().items()} == {k: tuple(v.shape) for k, v in want.items()}
    assert sum(p.numel() for p in pv.PhotoVerseAdapter(num_tokens=5).parameters()) == 28_904_960   # SURVEY 2 (measured)
    if ref_loader.reference_available():
        ref = ref_loader.load_reference_adapter_module().PhotoVerseAdapter(num_tokens=3)
        assert list(ref.state_dict().keys()) == list(ad.state_dict().keys())


def test_fusion_rule_consumes_exactly_one_rand_per_grad_call():
    p = pv.PhotoVerseAttnProcessor2_0(320, 768)
    torch.manual_seed(123)
    expect = [torch.rand(1).item() for _ in range(4)]
    torch.manual_seed(123)
    with torch.enable_grad():
        got = [p._fusion_weights() for _ in range(3)]
    for u, w in zip(expect, got):
        assert w == ((2.0, 0.0) if u < 1 / 3 else (0.0, 2.0) if u > 2 / 3 else (1.0, 1.0))
    assert torch.rand(1).item() == expect[3]          # RNG stream stays aligned with the reference's
    torch.manual_seed(123)
    with torch.no_grad():
        assert p._fusion_weights() == (1.0, 1.0)
    assert torch.rand(1).item() == expect[0]          # no draw without grad (attention_processor.py:411)


def test_install_on_sd15_unet_and_regulariser_gather():
    unet = UNetSD15()
    assert len(unet.attn_processors) == 32
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
    procs = unet.attn_processors
    attn2 = {k: v for k, v in procs.items() if k.endswith("attn2.processor")}
    assert sorted(attn2) == sorted(f"{p}.transformer_blocks.0.attn2.processor" for p in SD15_ATTN2)
    widths = {k: v.hidden_size for k, v in attn2.items()}
    assert widths["down_blocks.0.attentions.0.transformer_blocks.0.attn2.processor"] == 320
    assert widths["down_blocks.1.attentions.1.transformer_blocks.0.attn2.processor"] == 640
    assert widths["mid_block.attentions.0.transformer_blocks.0.attn2.processor"] == 1280
    assert widths["up_blocks.1.attentions.2.transformer_blocks.0.attn2.processor"] == 1280
    assert widths["up_blocks.3.attentions.0.transformer_blocks.0.attn2.processor"] == 320
    assert all(not isinstance(v, torch.nn.Module) for k, v in procs.items() if k.endswith("attn1.processor"))
    # processor weights live in unet.state_dict() under the reference's key names (modeling_utils.py:33-37)
    keys = [k for k in unet.state_dict() if "attn2" in k and ("processor" in k or "to_q" in k or "to_k" in k or "to_v" in k)]
    assert "mid_block.attentions.0.transformer_blocks.0.attn2.processor.to_k_ip.0.weight" in keys
    assert sum(unet.state_dict()[k].numel() for k in keys if "processor" in k) == 19_169_280         # SURVEY 8 a2
    for i, p in enumerate(attn2.values()):
        p.to_v_ip_norm = torch.full((2, 8, 5, 1), float(i))
    g = pv.get_visual_cross_attention_values_norm(unet)
    assert g.shape == (2, 16 * 8 * 5)
    pv.set_cross_attention_layers_to_train(unet)
    with pytest.raises(ValueError, match="number of processors"):
        unet.set_attn_processor({"x": None})


def test_unet_forward_shapes_cpu_tiny():
    """Backbone wiring (skip connections, up/down sampling) on a 2-level variant with stock processors."""
    unet = UNetSD15(block_out_channels=(32, 64), layers_per_block=1, heads=4, cross_attention_dim=16)
    x = torch.randn(2, 4, 16, 16)
    y = unet(x, torch.tensor([10.0]), encoder_hidden_states=torch.randn(2, 7, 16)).sample
    assert y.shape == x.shape and torch.isfinite(y).all()


def test_lora_injection_matches_peft_layout():
    unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet)
    inject_lora(unet, r=8, lora_alpha=1.0)
    names = [n for n, m in unet.named_modules() if isinstance(m, LoraLinear)]
    assert names and all(n.split(".")[-2] == "attn2" and n.split(".")[-1] in ("to_q", "to_k", "to_v") for n in names)
    sd = unet.state_dict()
    k = "mid_block.attentions.0.transformer_blocks.0.attn2.to_q"
    assert f"{k}.base_layer.weight" in sd and f"{k}.lora_A.default.weight" in sd and f"{k}.lora_B.default.weight" in sd
    assert sd[f"{k}.lora_A.default.weight"].shape == (8, 640) and sd[f"{k}.lora_B.default.weight"].abs().sum() == 0
    trainable = [n for n, p in unet.named_parameters() if p.requires_grad]
    assert trainable and all("lora_" in n for n in trainable)          # peft freezes the rest (SURVEY D8)
    w, A, B, s, p = linear_parts(unet.mid_block.attentions[0].transformer_blocks[0].attn2.to_q)
    assert w.shape == (640, 640) and A.shape == (8, 640) and B.shape == (640, 8) and s == 1 / 8 and p == 0.0
    n_lora = sum(p.numel() for n, p in UNetSD15_lora_params().items())
    assert n_lora == 595_968                                            # SURVEY 8 a5 (r = 8, 16 layers)


def test_lora_dropout_routing_follows_the_train_toggle():
    """peft applies `lora_dropout` only in training mode; the reference switches the attn2 modules to train() with
    `set_cross_attention_layers_to_train` (models/unet.py:50-53, train.py:462).  The processor must take the un-merged
    path exactly then."""
    unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet)
    inject_lora(unet, r=8, lora_dropout=0.1)
    unet.eval()
    attn = unet.mid_block.attentions[0].transformer_blocks[0].attn2
    proc = attn.processor
    assert linear_parts(attn.to_q)[4] == 0.0 and not proc.lora_dropout_active(attn)        # eval: nn.Dropout is the identity
    pv.set_cross_attention_layers_to_train(unet)
    assert attn.to_q.training and linear_parts(attn.to_q)[4] == pytest.approx(0.1)
    assert proc.lora_dropout_active(attn)
    attn1 = unet.mid_block.attentions[0].transformer_blocks[0].attn1
    assert not attn1.training                                                              # only attn2 is switched
    plain = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(plain)
    inject_lora(plain, r=8)                                                                # p = 0: nn.Identity
    pv.set_cross_attention_layers_to_train(plain)
    a2 = plain.mid_block.attentions[0].transformer_blocks[0].attn2
    assert not a2.processor.lora_dropout_active(a2)


def UNetSD15_lora_params():
    unet = UNetSD15()
    inject_lora(unet, r=8)
    return {n: p for n, p in unet.named_parameters() if "lora_" in n}


def test_ddim_schedule():
    s = make_ddim_schedule(50)
    assert len(s.timesteps) == 50 and s.timesteps[0] == 981 and s.timesteps[-1] == 1
    assert all(a > b for a, b in zip(s.timesteps, s.timesteps[1:]))
    # one step with eps = 0 only rescales x; with the true noise it recovers x0 on the last step
    import numpy as np
    betas = np.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000) ** 2
    ac = np.cumprod(1 - betas)
    t = s.timesteps[-1]
    x0, eps = 0.7, -1.3
    xt = ac[t] ** 0.5 * x0 + (1 - ac[t]) ** 0.5 * eps
    x_prev = s.c_x[-1] * xt + s.c_eps[-1] * eps
    assert abs(x_prev - (ac[0] ** 0.5 * x0 + (1 - ac[0]) ** 0.5 * eps)) < 1e-9


def test_checkpoint_wire_format_round_trip(tmp_path):
    """models/modeling_utils.py:13-50: dict keys, the attn2 key filter, peft-style LoRA keys, lora_config re-injection."""
    from photoverse_b200.checkpoint import cross_attention_state_dict, load_photoverse_model, save_progress
    torch.manual_seed(0)
    unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet)
    inject_lora(unet, r=4, lora_alpha=2.0)
    ia, ta = pv.PhotoVerseAdapter(num_tokens=2), pv.PhotoVerseAdapter(num_tokens=2)
    with torch.no_grad():
        for n, p in unet.named_parameters():
            if "lora_B" in n:
                p.normal_()
    cfg = {"r": 4, "lora_alpha": 2.0, "lora_dropout": 0.0, "target_modules": ["attn2.to_k", "attn2.to_v", "attn2.to_q"]}
    path = save_progress(ia, ta, unet, str(tmp_path), step=7, lora_config=cfg)
    assert path.endswith("photoverse_000007.pt")
    sd = torch.load(path, map_location="cpu")
    assert set(sd) == {"image_adapter", "text_adapter", "cross_attention_adapter", "lora_config"}
    keys = list(sd["cross_attention_adapter"])
    assert keys == list(cross_attention_state_dict(unet)) and all("attn2" in k for k in keys)
    k = "mid_block.attentions.0.transformer_blocks.0.attn2"
    for suffix in ("processor.to_k_ip.0.weight", "processor.to_v_ip.0.weight", "to_q.base_layer.weight",
                   "to_q.lora_A.default.weight", "to_q.lora_B.default.weight", "to_v.lora_B.default.weight"):
        assert f"{k}.{suffix}" in keys
    assert not any("to_out" in x or "attn1" in x for x in keys)
    # load into a fresh model WITHOUT LoRA wrappers: the stored lora_config re-injects them (modeling_utils.py:15-18)
    torch.manual_seed(1)
    unet2 = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet2)
    ia2, ta2 = pv.PhotoVerseAdapter(num_tokens=2), pv.PhotoVerseAdapter(num_tokens=2)
    _, _, unet2, cfg2 = load_photoverse_model(path, ia2, ta2, unet2)
    assert cfg2 == cfg
    a, b = cross_attention_state_dict(unet), cross_attention_state_dict(unet2)
    assert list(a) == list(b) and all(torch.equal(a[x], b[x]) for x in a)
    assert all(torch.equal(p, q) for p, q in zip(ia.state_dict().values(), ia2.state_dict().values()))
    assert save_progress(ia, ta, unet, str(tmp_path)).endswith("photoverse.pt")


def test_checkpoint_written_by_the_reference_loads(tmp_path):
    """A file written by the VERBATIM reference ``save_progress`` (modeling_utils.py:29-50: its key filter, its
    ``lora_config.to_dict()`` with a peft PeftType enum member and a ``set``) loads into the B200 classes under
    torch.load's weights-only rules; and a file written here is read by the verbatim reference loader.  Runs the
    upstream functions themselves, so it needs PHOTOVERSE_REFERENCE_ROOT set to a checkout of the upstream project."""
    from oracle import ref_loader
    if not ref_loader.reference_available():
        pytest.skip("PHOTOVERSE_REFERENCE_ROOT does not name a checkout of the upstream project")
    from types import SimpleNamespace
    from photoverse_b200.checkpoint import cross_attention_state_dict, load_photoverse_model, save_progress
    ref_save, ref_load, RefLoraConfig = ref_loader.load_reference_checkpoint_fns()
    targets = ["attn2.to_k", "attn2.to_v", "attn2.to_q"]

    def fresh(seed, lora):
        torch.manual_seed(seed)
        u = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
        pv.set_visual_cross_attention_adapter(u)
        if lora:
            inject_lora(u, r=4, lora_alpha=2.0)
            with torch.no_grad():
                for n, p in u.named_parameters():
                    if "lora_B" in n:
                        p.normal_()
        return u, pv.PhotoVerseAdapter(num_tokens=2), pv.PhotoVerseAdapter(num_tokens=2)

    # reference writes -> we read
    unet, ia, ta = fresh(0, lora=True)
    accel = SimpleNamespace(unwrap_model=lambda m: m)
    cfg = RefLoraConfig(r=4, lora_alpha=2.0, lora_dropout=0.1, target_modules=targets)
    opt = torch.optim.AdamW(ia.parameters(), lr=1e-4)
    ref_save(ia, ta, unet, accel, str(tmp_path), step=3, lora_config=cfg, optimizer=opt)
    path = str(tmp_path / "photoverse_000003.pt")
    with pytest.raises(Exception):                     # the raw file is NOT loadable with torch's default rules ...
        torch.load(path, map_location="cpu")
    unet2, ia2, ta2 = fresh(1, lora=False)             # ... and carries the enum + set; no LoRA wrappers yet
    _, _, unet2, cfg2 = load_photoverse_model(path, ia2, ta2, unet2)
    assert cfg2["r"] == 4 and cfg2["lora_alpha"] == 2.0 and cfg2["lora_dropout"] == 0.1 and cfg2["peft_type"] == "LORA"
    assert cfg2["target_modules"] == sorted(targets)
    a, b = cross_attention_state_dict(unet), cross_attention_state_dict(unet2)
    assert list(a) == list(b) and len(a) > 0 and all(torch.equal(a[k], b[k]) for k in a)
    assert all(torch.equal(p, q) for p, q in zip(ta.state_dict().values(), ta2.state_dict().values()))
    from photoverse_b200.lora import linear_parts
    mod = unet2.mid_block.attentions[0].transformer_blocks[0].attn2.to_q
    assert linear_parts(mod.train())[3] == 0.5 and linear_parts(mod)[4] == pytest.approx(0.1)   # scaling alpha / r, dropout p

    # we write -> the reference reads (its LoraConfig(**cfg) + inject + strict=False load)
    ours = save_progress(ia, ta, unet, str(tmp_path), step=4, lora_config=cfg)
    assert isinstance(torch.load(ours, map_location="cpu")["lora_config"]["target_modules"], list)   # plain types
    unet3, ia3, ta3 = fresh(2, lora=False)
    _, _, unet3, cfg3 = ref_load(ours, ia3, ta3, unet3)
    assert cfg3.r == 4 and set(cfg3.target_modules) == set(targets)
    c = cross_attention_state_dict(unet3)
    assert list(a) == list(c) and all(torch.equal(a[k], c[k]) for k in a)


def test_dpmpp_2m_schedule_is_exact_for_a_perfect_denoiser():
    """DPM-Solver++(2M) (reference sampler, infer.py:39-40): with the exact epsilon of a fixed x0 every step must land on
    alpha_t x0 + sigma_t n exactly (the solver integrates the data-prediction ODE exactly for constant x0), for the
    first-order start, the 2M steps and the final step.  diffusers' default ``final_sigmas_type="zero"`` closes the grid
    with sigma = 0: the last step is first-order for EVERY N and returns the data prediction itself; the coefficients of
    that step are pinned to the closed form of diffusers' first-order update at (alpha, sigma) = (1, 0)."""
    import numpy as np
    from photoverse_b200.host.dpm_solver import make_dpmpp_2m_schedule
    betas = np.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000) ** 2
    ac = np.cumprod(1 - betas)
    for final in ("zero", "sigma_min"):
        for n in (10, 25, 50):
            s = make_dpmpp_2m_schedule(n, final_sigmas_type=final)
            assert len(s.timesteps) == n and s.timesteps[0] == 999 and all(a > b for a, b in zip(s.timesteps, s.timesteps[1:]))
            assert all(np.isfinite(v) for v in s.cx + s.c0 + s.c0p + s.kx + s.ke)
            assert s.c0p[0] == 0.0 and all(c != 0.0 for c in s.c0p[1:-1])
            if final == "zero":
                assert (s.cx[-1], s.c0[-1], s.c0p[-1]) == (0.0, 1.0, 0.0)       # x_N = x0 prediction, first order
            else:
                assert (s.c0p[-1] == 0.0) == (n < 15)
            x0, noise = 0.7, -1.3
            nodes = s.timesteps + [0]
            x = ac[nodes[0]] ** 0.5 * x0 + (1 - ac[nodes[0]]) ** 0.5 * noise
            x0_prev = None
            for i in range(n):
                t = nodes[i]
                eps = (x - ac[t] ** 0.5 * x0) / (1 - ac[t]) ** 0.5              # the perfect epsilon-prediction
                d = s.kx[i] * x + s.ke[i] * eps
                assert abs(d - x0) < 1e-9
                x = s.cx[i] * x + s.c0[i] * d + (s.c0p[i] * x0_prev if s.c0p[i] != 0.0 else 0.0)
                x0_prev = d
                if final == "zero" and i == n - 1:
                    assert abs(x - x0) < 1e-9                                   # sigma = 0: no residual noise
                else:
                    tn = nodes[i + 1]
                    assert abs(x - (ac[tn] ** 0.5 * x0 + (1 - ac[tn]) ** 0.5 * noise)) < 1e-9
    # first-order update of diffusers at the terminal node: x_t = (sigma_t / sigma_s) x - alpha_t (exp(-h) - 1) x0 with
    # sigma_t = 0, alpha_t = 1, h = lambda_t - lambda_s = +inf  ->  0 * x + 1 * x0
    assert (0.0 / (1 - ac[20]) ** 0.5, -1.0 * (np.exp(-np.inf) - 1.0)) == (0.0, 1.0)


def test_backbone_epilogue_helpers_keep_the_stock_ops_off_the_gpu_path():
    """`group_norm_act` / `layer_norm` / GEGLU of the host UNet (photoverse_b200/host/unet_sd15.py) are the stock PyTorch ops
    whenever the pv_backbone.cu kernels do not apply (CPU tensors here); the per-model switch marks exactly the norm / GEGLU
    modules."""
    import torch.nn.functional as F
    from photoverse_b200.host import unet_sd15 as U
    torch.manual_seed(0)
    norm = torch.nn.GroupNorm(4, 16)
    x = torch.randn(2, 16, 5, 3)
    add = torch.randn(2, 16)
    assert torch.equal(U.group_norm_act(norm, x, True), F.silu(norm(x)))
    assert torch.equal(U.group_norm_act(norm, x, False), norm(x))
    assert torch.allclose(U.group_norm_act(norm, x, True, add), F.silu(norm(x + add[:, :, None, None])))
    ln = torch.nn.LayerNorm(16)
    t = torch.randn(2, 7, 16)
    assert torch.equal(U.layer_norm(ln, t), ln(t))
    ge = U.GEGLU(16, 32)
    h = ge.proj(t)
    assert torch.equal(ge(t), h[..., :32] * F.gelu(h[..., 32:]))
    unet = UNetSD15(block_out_channels=(32, 64), layers_per_block=1, heads=2, cross_attention_dim=16, sample_size=8)
    marked = [m for m in unet.set_fused_epilogues(False).modules() if getattr(m, "_pv_fused", None) is False]
    expect = [m for m in unet.modules() if isinstance(m, (torch.nn.GroupNorm, torch.nn.LayerNorm, U.GEGLU))]
    assert marked and len(marked) == len(expect)
    # a resnet block on the stock path: conv bias and the time-embedding term are added before norm2, as in diffusers
    blk = U.ResnetBlock2D(16, 32, 8, groups=4)
    xin, temb = torch.randn(2, 16, 4, 4), torch.randn(2, 8)
    hh = blk.conv1(F.silu(blk.norm1(xin))) + blk.time_emb_proj(F.silu(temb))[:, :, None, None]
    ref = blk.conv_shortcut(xin) + blk.conv2(F.silu(blk.norm2(hh)))
    assert torch.allclose(blk(xin, temb), ref, atol=1e-6)
