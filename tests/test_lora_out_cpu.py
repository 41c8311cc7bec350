"""CPU: LoRA on the cross-attention out projection (``attn2.to_out.0``) -- injection, the checkpoint keys and the test
reference of peft 0.10.0 ``lora.Linear`` at attention_processor.py:423 (tests/lora_out_reference.py)."""
import pytest
import torch

import photoverse_b200 as pv
from oracle import cases, detgen
from oracle.processor_oracle import LoraWeights, dual_branch_attention
from photoverse_b200.host.unet_sd15 import UNetSD15
from photoverse_b200.lora import DEFAULT_TARGETS, LoraLinear, inject_lora, linear_parts
from tests.lora_out_reference import dual_branch_attention_out_lora

OUT_TARGETS = DEFAULT_TARGETS + ("attn2.to_out.0",)


def test_inject_wraps_exactly_the_attn2_out_projections():
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet)
    inject_lora(unet, r=8, target_modules=OUT_TARGETS)
    wrapped = [n for n, m in unet.named_modules() if isinstance(m, LoraLinear)]
    out = [n for n in wrapped if n.endswith("to_out.0")]
    assert len(out) == 16 and all(n.endswith("attn2.to_out.0") for n in out)
    assert len(wrapped) == 4 * 16 and not any("attn1" in n for n in wrapped)
    attn = unet.mid_block.attentions[0].transformer_blocks[0].attn2
    w, A, B, s, p = linear_parts(attn.to_out[0])
    assert w.shape == (1280, 1280) and A.shape == (8, 1280) and B.shape == (1280, 8) and s == 1 / 8 and p == 0.0
    assert attn.to_out[0].bias is attn.to_out[0].base_layer.bias and not attn.to_out[0].bias.requires_grad
    assert isinstance(unet.mid_block.attentions[0].transformer_blocks[0].attn1.to_out[0], torch.nn.Linear)


def test_lora_dropout_on_the_out_projection_selects_the_unmerged_path():
    unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(unet)
    inject_lora(unet, r=4, target_modules=("attn2.to_out.0",), lora_dropout=0.1)
    unet.eval()
    attn = unet.mid_block.attentions[0].transformer_blocks[0].attn2
    assert not attn.processor.lora_dropout_active(attn)
    pv.set_cross_attention_layers_to_train(unet)
    assert attn.processor.lora_dropout_active(attn)


def _unet_with_out_lora(seed, lora):
    torch.manual_seed(seed)
    u = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
    pv.set_visual_cross_attention_adapter(u)
    if lora:
        inject_lora(u, r=4, lora_alpha=2.0, target_modules=OUT_TARGETS)
        with torch.no_grad():
            for n, p in u.named_parameters():
                if "lora_B" in n:
                    p.normal_()
    return u, pv.PhotoVerseAdapter(num_tokens=2), pv.PhotoVerseAdapter(num_tokens=2)


def test_checkpoint_round_trip_carries_the_out_projection_lora(tmp_path):
    from photoverse_b200.checkpoint import cross_attention_state_dict, load_photoverse_model, save_progress
    unet, ia, ta = _unet_with_out_lora(0, lora=True)
    cfg = {"r": 4, "lora_alpha": 2.0, "lora_dropout": 0.0, "target_modules": list(OUT_TARGETS)}
    path = save_progress(ia, ta, unet, str(tmp_path), step=1, lora_config=cfg)
    keys = list(torch.load(path, map_location="cpu")["cross_attention_adapter"])
    k = "mid_block.attentions.0.transformer_blocks.0.attn2.to_out.0"
    for suffix in ("base_layer.weight", "base_layer.bias", "lora_A.default.weight", "lora_B.default.weight"):
        assert f"{k}.{suffix}" in keys
    assert sum(x.endswith("to_out.0.lora_B.default.weight") for x in keys) == 4      # one per attn2 layer
    assert not any("attn1" in x for x in keys)
    unet2, ia2, ta2 = _unet_with_out_lora(1, lora=False)
    _, _, unet2, cfg2 = load_photoverse_model(path, ia2, ta2, unet2)
    assert cfg2 == cfg
    a, b = cross_attention_state_dict(unet), cross_attention_state_dict(unet2)
    assert list(a) == list(b) and all(torch.equal(a[x], b[x]) for x in a)
    assert isinstance(unet2.mid_block.attentions[0].transformer_blocks[0].attn2.to_out[0], LoraLinear)


def test_checkpoint_keys_without_an_out_projection_lora_are_unchanged():
    from photoverse_b200.checkpoint import cross_attention_state_dict
    unet, _, _ = _unet_with_out_lora(0, lora=False)
    inject_lora(unet, r=4)
    keys = list(cross_attention_state_dict(unet))
    want = [k for k in unet.state_dict() if "attn2" in k and any(t in k for t in ("processor", "to_q", "to_k", "to_v"))]
    assert keys == want and not any("to_out" in k for k in keys)


def _out_lora_case(r, p):
    case = cases.ProcCase("out_cpu", B=2, S=40, C=320, Li=3, lora_r=4, seed=41)
    w = cases.proc_weights(case, torch.float64)
    w.lora["to_out"] = LoraWeights(A=detgen.uniform_linear(r, case.C, 4190, torch.float64),
                                   B=detgen.uniform((case.C, r), 4191, -0.2, 0.2, torch.float64), scaling=2.0 / r)
    x, text, img = (t.double() for t in cases.proc_inputs(case, torch.float64))
    g = torch.Generator().manual_seed(7)
    mask = torch.rand(case.B, case.S, case.C, generator=g) >= p
    return case, w, x, text, img, mask


@pytest.mark.parametrize("r,p", [(4, 0.0), (16, 0.1)])
def test_out_lora_reference_is_peft_linear(r, p):
    """The test reference of the out-projection LoRA against peft's formula written out in fp64:
    y = O Wo^T + bo + s B_o A_o dropout(O), with O recovered from the plain oracle's output by solving O Wo^T = y - bo."""
    case, w, x, text, img, mask = _out_lora_case(r, p)
    y, vn = dual_branch_attention_out_lora(x, text, img, w, 1.0, 1.0, {"to_out": (mask, p)} if p else None)
    plain = w.to()
    lo = plain.lora.pop("to_out")
    y_plain, vn_plain = dual_branch_attention(x, text, img, plain)
    o = torch.linalg.solve(w.to_out_w, (y_plain - w.to_out_b).reshape(-1, case.C).t()).t().reshape(y.shape)
    od = o * mask / (1.0 - p) if p else o
    want = y_plain + lo.scaling * (od @ lo.A.t()) @ lo.B.t()
    assert torch.allclose(y, want, rtol=1e-9, atol=1e-9)
    assert torch.equal(vn, vn_plain) and (y - y_plain).abs().max() > 1e-3
    # without a to_out entry it is the oracle itself
    y0, vn0 = dual_branch_attention_out_lora(x, text, img, plain)
    assert torch.equal(y0, y_plain) and torch.equal(vn0, vn_plain)
