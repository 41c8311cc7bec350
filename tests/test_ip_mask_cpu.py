"""CPU: regional identity masks (diffusers' ``ip_adapter_masks``) -- the downsample restatement against diffusers' formula,
the processor's validation (raised before any CUDA work) and the C ABI declarations of the masked entry points."""
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

from tests.ip_mask_reference import downsample, grid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ("pv_ip_mask_downsample", "pv_dual_attn_masked_fwd", "pv_dual_attn_masked_core_fwd",
               "pv_dual_attn_masked_bwd")


def _diffusers_downsample(mask, batch_size, num_queries, value_embed_dim):
    """diffusers 0.27.2 IPAdapterMaskProcessor.downsample, written out as published."""
    o_h = mask.shape[1]
    o_w = mask.shape[2]
    ratio = o_w / o_h
    mask_h = int(math.sqrt(num_queries / ratio))
    mask_h = int(mask_h) + int((num_queries % int(mask_h)) != 0)
    mask_w = num_queries // mask_h
    mask_downsample = F.interpolate(mask.unsqueeze(0), size=(mask_h, mask_w), mode="bicubic").squeeze(0)
    if mask_downsample.shape[0] < batch_size:
        mask_downsample = mask_downsample.repeat(batch_size, 1, 1)
    mask_downsample = mask_downsample.view(mask_downsample.shape[0], -1)
    downsampled_area = mask_h * mask_w
    if downsampled_area < num_queries:
        mask_downsample = F.pad(mask_downsample, (0, num_queries - mask_downsample.shape[1]), value=0.0)
    if downsampled_area > num_queries:
        mask_downsample = mask_downsample[:, :num_queries]
    return mask_downsample.view(mask_downsample.shape[0], mask_downsample.shape[1], 1).repeat(1, 1, value_embed_dim)


@pytest.mark.parametrize("mb,H,W,S,B", [
    (1, 64, 64, 4096, 2), (1, 512, 512, 1024, 3), (2, 96, 64, 9216, 2),     # square, mask batch B, portrait
    (1, 64, 96, 256, 4), (1, 77, 130, 144, 1),                               # landscape, odd sizes
    (1, 64, 64, 200, 2),                                                     # S not a square: zero padding
])
def test_downsample_equals_diffusers(mb, H, W, S, B):
    g = torch.Generator().manual_seed(H * W + S)
    mask = torch.rand(mb, H, W, generator=g, dtype=torch.float64)
    ref = _diffusers_downsample(mask, B, S, 3)
    assert torch.equal(ref[..., 0], ref[..., 2])
    got = downsample(mask, B, S)
    assert got.shape == (B, S)
    assert torch.allclose(got, ref[..., 0], rtol=0, atol=1e-12)
    mh, mw = grid(S, H, W)
    if mh * mw < S:
        assert (got[:, mh * mw:] == 0).all()


def test_grid_pads_when_the_grid_does_not_cover_s():
    assert grid(200, 64, 64) == (15, 13)           # 195 < 200 rows: five zero rows
    assert grid(4096, 64, 64) == (64, 64)
    assert grid(9216, 768, 768) == (96, 96)


def _layer():
    from photoverse_b200.attention_processor import PhotoVerseAttnProcessor2_0
    from photoverse_b200.host.unet_sd15 import Attention
    attn = Attention(320, 768, 8)
    attn.set_processor(PhotoVerseAttnProcessor2_0(hidden_size=320, cross_attention_dim=768, num_tokens=(5,)))
    return attn


@pytest.mark.parametrize("masks,exc,msg", [
    ([torch.ones(1, 1, 8, 8), torch.ones(1, 1, 8, 8)], ValueError, "Length of ip_adapter_masks"),
    ([], ValueError, "Length of ip_adapter_masks"),
    ([torch.ones(1, 8, 8)], ValueError, "should be a tensor with shape"),
    (["mask"], ValueError, "should be a tensor with shape"),
    ([torch.ones(1, 2, 8, 8)], NotImplementedError, "several images per adapter"),
    ([torch.ones(1, 0, 8, 8)], ValueError, "Number of masks"),
    ([torch.ones(3, 1, 8, 8)], ValueError, "mask batch"),
    ([torch.ones(1, 1, 8, 8, dtype=torch.int64)], TypeError, "floating-point"),
    (torch.ones(2, 1, 8, 8), ValueError, "Length of ip_adapter_masks"),        # tensor form: two adapters' masks
])
def test_processor_validation_before_any_cuda_work(masks, exc, msg):
    """Each error is raised from CPU tensors: nothing reaches the native library first."""
    attn = _layer()
    x = torch.zeros(2, 64, 320)
    ehs = (torch.zeros(2, 77, 768), torch.zeros(2, 5, 768))
    with pytest.raises(exc, match=msg):
        attn(x, encoder_hidden_states=ehs, ip_adapter_masks=masks)


def test_tensor_form_and_list_form_pass_validation():
    """A [1, 1, H, W] tensor (diffusers' tensor form) and a one-element list both reach the device check."""
    for masks in (torch.ones(1, 1, 8, 8), [torch.ones(2, 1, 8, 8)]):
        attn = _layer()
        with pytest.raises(RuntimeError, match="CUDA only"):
            attn(torch.zeros(2, 64, 320), encoder_hidden_states=(torch.zeros(2, 77, 768), torch.zeros(2, 5, 768)),
                 ip_adapter_masks=masks)


def test_attention_mask_is_still_refused():
    attn = _layer()
    with pytest.raises(NotImplementedError, match="attention_mask"):
        attn(torch.zeros(2, 64, 320), encoder_hidden_states=(torch.zeros(2, 77, 768), torch.zeros(2, 5, 768)),
             attention_mask=torch.ones(2, 64))


def test_new_symbols_in_header_and_signatures():
    from photoverse_b200 import _lib
    with open(os.path.join(ROOT, "include", "photoverse_b200.h")) as f:
        hdr = f.read()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\bint {name}\(", hdr), name
        assert name in _lib._SIGNATURES, name
    assert "#define PV_ABI_VERSION 2" in hdr


def test_masked_backward_rejects_f16_by_name():
    from photoverse_b200 import _lib
    lib = _lib.lib()
    rc = lib.pv_dual_attn_masked_bwd(_lib.PV_F16, *([None] * 7), 1, 256, 320, 8, 77, 5, 1.0, 1.0, None, None)
    assert rc == 3                                                      # PV_ERR_UNSUPPORTED
    msg = lib.pv_last_error().decode()
    assert "pv_dual_attn_masked_bwd" in msg and "PV_F16" in msg, msg


def test_downsample_rejects_a_mask_without_a_grid():
    """A mask far wider than S rows has no diffusers grid (int(sqrt(S / ratio)) == 0): PV_ERR_INVALID, no launch."""
    from photoverse_b200 import _lib
    lib = _lib.lib()
    assert lib.pv_ip_mask_downsample(None, 1, 8, 8, None, 1, 64, None) == 1
    import ctypes
    buf = ctypes.c_void_p(16)          # never dereferenced: the shape check fails first
    assert lib.pv_ip_mask_downsample(buf, 1, 1, 4096, buf, 1, 64, None) == 1
    assert "no query grid" in lib.pv_last_error().decode()
    assert lib.pv_ip_mask_downsample(buf, 3, 8, 8, buf, 2, 64, None) == 1
