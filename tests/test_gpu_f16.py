"""GPU (B200): the float16 inference path -- processor and adapters of a model run in float16 -- against the fp64 oracle.

The fp16 kernels round at the points where the bf16 kernels do (Q in TMEM, P for the PV MMA, O at the drain, Y after the
bias), so with 3 more mantissa bits their error on the same inputs must be below the bf16 path's: a bf16 computation
behind a cast would not pass that check.
"""
import numpy as np
import pytest
import torch

from oracle import adapter_oracle, cases
from oracle.processor_oracle import dual_branch_attention
from tests.helpers import build_product_layer, golden

pytestmark = pytest.mark.gpu


def _call(attn, x, text, img, dtype, dev):
    with torch.no_grad():
        return attn(x.to(dev, dtype), encoder_hidden_states=(text.to(dev, dtype), img.to(dev, dtype)))


def _oracle64(case, x, text, img, dev):
    w = cases.proc_weights(case).to(dtype=torch.float64, device=dev)
    with torch.no_grad():
        return dual_branch_attention(x.to(dev, torch.float64), text.to(dev, torch.float64), img.to(dev, torch.float64), w)


# the four SD-1.5 attn2 layer shapes (S, C) at latent 64^2, a ragged S, Li in {1, 5, 16}, merged LoRA on to_q / to_k / to_v
SHAPES = [(2, 4096, 320, 1, 0), (2, 1024, 640, 5, 0), (2, 256, 1280, 16, 0), (2, 64, 1280, 5, 0),
          (3, 200, 320, 16, 4), (2, 330, 640, 1, 8), (1, 384, 1280, 5, 4), (2, 128, 320, 5, 4), (2, 100, 640, 16, 0)]


@pytest.mark.parametrize("fuse", [1, 2, 0], ids=["default", "one-launch", "attention+gemm"])
@pytest.mark.parametrize("B,S,C,Li,r", SHAPES, ids=[f"B{b}_S{s}_C{c}_Li{li}_r{r}" for b, s, c, li, r in SHAPES])
def test_processor_f16_vs_fp64_oracle(cuda_device, fuse, B, S, C, Li, r):
    from photoverse_b200 import _lib, ops
    if fuse != 1 and S <= 128:
        pytest.skip("S <= 128 has a single launch policy (attention kernel + out-projection GEMM)")
    case = cases.ProcCase(f"f16_{S}_{C}", B=B, S=S, C=C, Li=Li, lora_r=r, seed=90 + Li + r)
    attn, proc = build_product_layer(case, cuda_device)
    x, text, img = cases.proc_inputs(case, torch.float32)
    y_ref, vn_ref = _oracle64(case, x, text, img, cuda_device)
    _lib.set_option("fuse_out", fuse)
    try:
        y16 = _call(attn, x, text, img, torch.float16, cuda_device)
        vn16 = proc.to_v_ip_norm
        y16b = _call(attn, x, text, img, torch.float16, cuda_device)      # same row-block counters, same packed weights
        y_bf = _call(attn, x, text, img, torch.bfloat16, cuda_device)
    finally:
        _lib.set_option("fuse_out", 1)
    assert y16.dtype == torch.float16 and y16.shape == (B, S, C) and vn16.dtype == torch.float16
    assert torch.isfinite(y16).all()
    assert torch.equal(y16, y16b), "two fp16 calls differ"
    for buf in ops._SYNC.values():
        assert int(buf.abs().max().item()) == 0, "row-block counters must be zero after the call"
    e16 = (y16.double() - y_ref).abs().max().item()
    ebf = (y_bf.double() - y_ref).abs().max().item()
    print(f"max-abs vs fp64: fp16 {e16:.3e}  bf16 {ebf:.3e}  ratio {ebf / max(e16, 1e-30):.1f}")
    assert e16 <= 2e-2, f"fp16 max-abs {e16}"
    assert e16 < ebf, f"fp16 error {e16} not below the bf16 error {ebf}"
    assert (vn16.double() / vn_ref - 1.0).abs().max().item() <= 2e-3


def test_processor_f16_kv_cache_and_launches(cuda_device):
    """A cached fp16 call launches what a cached bf16 call launches (one kernel at C = 320, S > 128) and is bit-identical
    to the uncached call."""
    from photoverse_b200 import _lib
    case = cases.ProcCase("f16_cache", B=2, S=1024, C=320, Li=5, seed=7)
    attn, proc = build_product_layer(case, cuda_device)
    x, text, img = (t.to(cuda_device, torch.float16) for t in cases.proc_inputs(case, torch.float32))
    with torch.no_grad():
        y0 = attn(x, encoder_hidden_states=(text, img))
        proc.enable_kv_cache(True)
        attn(x, encoder_hidden_states=(text, img))
        n0 = _lib.launch_count()
        y1 = attn(x, encoder_hidden_states=(text, img))
        n1 = _lib.launch_count()
        proc.enable_kv_cache(False)
    assert torch.equal(y0, y1)
    assert n1 - n0 == 1


@pytest.mark.parametrize("case", [c for c in cases.ADAPTER_CASES if c.token_index in (0, "full")], ids=lambda c: c.name)
def test_adapter_f16_matches_golden(cuda_device, case):
    from photoverse_b200 import PhotoVerseAdapter
    g = golden(case.name)
    ad = PhotoVerseAdapter(num_tokens=case.T)
    ad.load_state_dict(adapter_oracle.make_state_dict(case.T, case.seed), strict=True)
    ad.to(cuda_device)
    err = {}
    for dt in (torch.float16, torch.bfloat16):
        embs = [e.to(cuda_device, dt) for e in cases.adapter_inputs(case)]
        with torch.no_grad():
            y = ad(embs, token_index=case.token_index)
        assert y.dtype == dt and y.shape == g["y"].shape
        err[dt] = np.abs(y.float().cpu().numpy() - g["y"]).max()
    print(f"adapter max-abs: fp16 {err[torch.float16]:.3e}  bf16 {err[torch.bfloat16]:.3e}")
    assert err[torch.float16] <= 4e-2
    assert err[torch.float16] < err[torch.bfloat16]


def test_f16_grad_mode_raises(cuda_device):
    from photoverse_b200 import PhotoVerseAdapter
    case = cases.ProcCase("f16_grad", B=1, S=256, C=320, Li=5, lora_r=4, seed=3)
    attn, proc = build_product_layer(case, cuda_device)
    x, text, img = (t.to(cuda_device, torch.float16) for t in cases.proc_inputs(case, torch.float32))
    with pytest.raises(NotImplementedError, match="bfloat16 or float32"):
        attn(x.requires_grad_(True), encoder_hidden_states=(text, img))
    ad = PhotoVerseAdapter(num_tokens=2).to(cuda_device)
    embs = [torch.randn(1, 257, 1024, device=cuda_device, dtype=torch.float16) for _ in range(2)]
    with pytest.raises(NotImplementedError, match="bfloat16 or float32"):
        ad(embs, token_index="full")


def test_f16_lora_dropout_raises(cuda_device):
    case = cases.ProcCase("f16_drop", B=1, S=256, C=320, Li=5, lora_r=4, seed=4)
    attn, proc = build_product_layer(case, cuda_device)
    attn.to_q.lora_dropout["default"] = torch.nn.Dropout(0.1)
    attn.train()
    x, text, img = (t.to(cuda_device, torch.float16) for t in cases.proc_inputs(case, torch.float32))
    with torch.no_grad(), pytest.raises(NotImplementedError, match="bfloat16 or float32"):
        attn(x, encoder_hidden_states=(text, img))


def test_half_unet_generation_matches_oracle_arm(cuda_device):
    """A .half() UNet through run_generation (K/V cache and CUDA graph on) and through the GenerationEngine vs the same
    loop around the oracle processors: final-latent cosine >= 0.999 (latent 32^2, batch 2)."""
    from tests.test_gpu_pipeline import _cos, _models
    from oracle.host_reference import clone_adapter_as_oracle, clone_with_oracle_processors
    from photoverse_b200.host.pipeline import GenerationEngine, run_generation, synthetic_inputs
    dtype = torch.float16
    unet, ia, ta = _models(cuda_device, torch.float32)
    unet.half(), ia.half(), ta.half()
    ref_unet = clone_with_oracle_processors(unet)
    ref_ia, ref_ta = clone_adapter_as_oracle(ia, cuda_device, dtype), clone_adapter_as_oracle(ta, cuda_device, dtype)
    inp = synthetic_inputs(2, 32, seed=21, device=cuda_device, dtype=dtype)
    lat = run_generation(unet, ia, ta, inp, num_steps=20, mode="batched", use_cuda_graph=True, kv_cache=True)
    ref = run_generation(ref_unet, ref_ia, ref_ta, inp, num_steps=20, mode="two_call", use_cuda_graph=False, kv_cache=False)
    assert lat.dtype == dtype and torch.isfinite(lat.float()).all()
    c = _cos(lat, ref)
    eng = GenerationEngine(unet, ia, ta, batch=2, latent=32, num_steps=20, dtype=dtype, device=cuda_device)
    eng.load_inputs(inp)
    e = eng.generate().clone()
    eng.close()
    ce = _cos(e, ref)
    print(f"fp16 UNet final-latent cosine: run_generation {c:.6f}  engine {ce:.6f}")
    assert c >= 0.999 and ce >= 0.999
