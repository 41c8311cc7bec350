"""CPU: the oracle restatement against the committed golden vectors (generated from the verbatim reference by
oracle/make_golden.py) and, when PHOTOVERSE_REFERENCE_ROOT names a checkout of the upstream project, against the live
reference."""
import numpy as np
import pytest
import torch

from oracle import adapter_oracle, cases, ref_loader
from oracle.processor_oracle import (dual_branch_attention, fusion_weights, gather_values_norm, processor_flops,
                                     segment_softmax_form)
from tests.helpers import golden, manifest


@pytest.mark.parametrize("case", cases.PROC_CASES, ids=lambda c: c.name)
def test_processor_oracle_matches_golden(case):
    g = golden(case.name)
    w = cases.proc_weights(case, torch.float32)
    x, text, img = cases.proc_inputs(case, torch.float32)
    with torch.no_grad():
        y, vn = dual_branch_attention(x, text, img, w, case.w_text, case.w_img)
        y2, vn2 = segment_softmax_form(x, text, img, w, case.w_text, case.w_img)
    # fp32 oracle vs fp64 reference run: the reference's own fp32-vs-fp64 deviation is ~5e-7 (manifest)
    assert np.abs(y.numpy() - g["y"]).max() <= 3e-6
    assert np.abs(vn.numpy() - g["vnorm"]).max() <= 3e-6
    assert np.abs(y2.numpy() - g["y"]).max() <= 3e-6
    assert np.abs(vn2.numpy() - g["vnorm"]).max() <= 3e-6
    assert y.shape == (case.B, case.S, case.C) and vn.shape == (case.B, case.H, case.Li, 1)


@pytest.mark.parametrize("case", cases.ADAPTER_CASES, ids=lambda c: c.name)
def test_adapter_oracle_matches_golden(case):
    g = golden(case.name)
    sd = adapter_oracle.make_state_dict(case.T, case.seed)
    embs = cases.adapter_inputs(case)
    with torch.no_grad():
        y = adapter_oracle.adapter_forward(embs, sd, case.token_index)
    assert np.abs(y.numpy() - g["y"]).max() <= 2e-5
    n_out = 1 if (case.token_index is not None and case.token_index != "full") else case.T
    assert y.shape == (case.B, n_out, 768)


def test_manifest_records_reference_noise_floor():
    m = manifest()
    assert set(c.name for c in cases.PROC_CASES + cases.ADAPTER_CASES) | {"inject_concept"} == set(m["cases"])
    for v in m["cases"].values():
        if v["kind"] != "inject":                       # the injection is a gather: exact, no noise floor to record
            assert v["ref_f32_vs_f64_maxabs"] < 2e-6


def _assert_rounds_to(y64, g32):
    """The golden vectors are the reference's fp64 run rounded to fp32: an fp64 result equal to that run within 1e-12
    lies within half an fp32 ulp of the stored value."""
    assert (np.abs(y64 - g32) <= 0.5 * np.spacing(np.abs(g32)) + 1e-12).all()


@pytest.mark.parametrize("case", cases.PROC_CASES[:3] + cases.PROC_CASES[4:7], ids=lambda c: c.name)
def test_processor_oracle_matches_live_reference(case):
    w = cases.proc_weights(case, torch.float64)
    x, text, img = cases.proc_inputs(case, torch.float64)
    with torch.no_grad():
        y, vn = dual_branch_attention(x, text, img, w, case.w_text, case.w_img)
    g = golden(case.name)
    _assert_rounds_to(y.numpy(), g["y"])
    _assert_rounds_to(vn.numpy(), g["vnorm"])
    if ref_loader.reference_available():
        from oracle.make_golden import run_reference_processor
        y_ref, n_ref = run_reference_processor(case, torch.float64)
        assert (y - y_ref).abs().max().item() <= 1e-12
        assert (vn - n_ref).abs().max().item() <= 1e-12


def test_adapter_oracle_matches_live_reference():
    case = cases.ADAPTER_CASES[3]
    sd = adapter_oracle.make_state_dict(case.T, case.seed, dtype=torch.float64)
    with torch.no_grad():
        y = adapter_oracle.adapter_forward(cases.adapter_inputs(case, torch.float64), sd, case.token_index)
    _assert_rounds_to(y.numpy(), golden(case.name)["y"])
    if ref_loader.reference_available():
        from oracle.make_golden import run_reference_adapter
        y_ref = run_reference_adapter(case, torch.float64)
        assert (y - y_ref).abs().max().item() <= 1e-11


def test_fusion_rule_table():
    # attention_processor.py:411-420
    assert fusion_weights(False, None) == (1.0, 1.0)
    assert fusion_weights(True, 0.2) == (2.0, 0.0)
    assert fusion_weights(True, 0.5) == (1.0, 1.0)
    assert fusion_weights(True, 0.9) == (0.0, 2.0)
    assert fusion_weights(True, 1 / 3) == (1.0, 1.0)       # boundaries belong to the "sum" branch
    assert fusion_weights(True, 2 / 3) == (1.0, 1.0)


def test_gather_values_norm_layout():
    # models/unet.py:38-47 -> [B, n_layers*H*Li]
    norms = [torch.full((2, 8, 5, 1), float(i)) for i in range(16)]
    out = gather_values_norm(norms)
    assert out.shape == (2, 16 * 8 * 5)
    assert out[0, 0] == 0 and out[0, 40] == 1 and out[1, -1] == 15


def test_flop_formula_matches_survey():
    # SURVEY.md 8(d): 2.188 / 2.054 / 2.108 / 0.769 GFLOP per layer at latent 64^2, B=1, Li=5
    for (S, C), want in (((4096, 320), 2.188), ((1024, 640), 2.054), ((256, 1280), 2.108), ((64, 1280), 0.769)):
        assert abs(processor_flops(1, S, C, 77, 5) / 1e9 - want) < 2e-3
    assert abs(adapter_oracle.adapter_flops(1, 1) / 1e9 - 1.482) < 1e-3


def test_inject_oracle_matches_golden_and_live_reference():
    """Concept-token injection (models/clip.py:17-24): oracle vs the committed output of the verbatim function, and vs
    the function itself when the reference is mounted."""
    import numpy as np
    import torch
    from oracle import clip_oracle, ref_loader
    from tests.helpers import golden
    x, c, idx = clip_oracle.inject_case()
    y = clip_oracle.inject_concept_embeddings(x, c, idx)
    g = golden("inject_concept")
    assert list(g["idx"]) == idx
    assert np.array_equal(y.numpy()[:, :, :32], g["y"])
    assert y.shape == x.shape
    for b, i in enumerate(idx):                       # structural properties of the reference rule
        assert torch.equal(y[b, :i], x[b, :i]) and torch.equal(y[b, i:i + 5], c[b])
        assert torch.equal(y[b, i + 5:], x[b, i + 1:i + 1 + (77 - 5 - i)])
    if ref_loader.reference_available():
        assert torch.equal(ref_loader.load_reference_inject_fn()(x, c, idx), y)


def test_lora_dropout_oracle_matches_torch_dropout_module():
    """peft's ``lora_B(lora_A(dropout(x))) * scaling`` with ``nn.Dropout`` (train.py:264-269, p = 0.1 by default): the
    oracle's explicit keep-mask form equals the module form when the mask comes from the same generator state."""
    import torch
    from oracle.processor_oracle import LoraWeights, lora_linear
    g = torch.Generator().manual_seed(4)
    x = torch.randn(3, 11, 32, generator=g, dtype=torch.float64)
    w = torch.randn(24, 32, generator=g, dtype=torch.float64)
    lw = LoraWeights(torch.randn(4, 32, generator=g, dtype=torch.float64),
                     torch.randn(24, 4, generator=g, dtype=torch.float64), 0.25)
    torch.manual_seed(123)
    ref = x @ w.t() + torch.nn.Dropout(0.1)(x) @ lw.A.t() @ lw.B.t() * lw.scaling
    torch.manual_seed(123)
    _, mask = torch.native_dropout(x, 0.1, True)
    assert 0.8 < mask.double().mean().item() < 0.97
    assert (lora_linear(x, w, lw, (mask, 0.1)) - ref).abs().max().item() <= 1e-12
    assert torch.equal(lora_linear(x, w, lw, None), x @ w.t() + x @ lw.A.t() @ lw.B.t() * lw.scaling)
