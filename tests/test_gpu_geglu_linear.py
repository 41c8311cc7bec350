"""GPU (B200): the GEGLU feed-forward projection in one launch (ops.linear_geglu, the CTA-pair GEMM of csrc/pv_gemm3.cu
with the GEGLU epilogue) against the two-launch sequence it replaces in the host UNet, F.linear -> ops.geglu."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# (M, C): the ff.proj shapes of a batch-8 latent-64 generation (16 rows), a ragged M, and the small M of the latent-32 UNet
SHAPES = [(65536, 320), (16384, 640), (4096, 1280), (1024, 1280), (2 * 1024 + 40, 320),
          (2048, 320), (512, 640), (128, 1280), (32, 1280)]


def _problem(device, M, C, seed):
    g = torch.Generator().manual_seed(seed)
    lin = torch.nn.Linear(C, 8 * C)
    with torch.no_grad():                       # default init, then h of rms ~1.5 like test_geglu_matches_torch
        lin.weight.mul_(2.6)
        lin.bias.normal_(0.0, 0.3, generator=g)
    lin = lin.to(device, torch.bfloat16)
    x = torch.randn(M, C, generator=g).to(device, torch.bfloat16)
    return x, lin.weight.detach(), lin.bias.detach()


@pytest.mark.parametrize("M,C", SHAPES, ids=[f"M{m}_C{c}" for m, c in SHAPES])
def test_linear_geglu_matches_the_two_launch_path(cuda_device, M, C):
    from photoverse_b200 import ops
    x, w, b = _problem(cuda_device, M, C, M + C)
    wp, bp = ops.pack_geglu_weight(w, b)
    with torch.no_grad():
        y = ops.linear_geglu(x, wp, bp)
        h = F.linear(x, w, b)
        ref = ops.geglu(h)
    assert y.shape == (M, 4 * C) and y.dtype == torch.bfloat16
    # same rounding points; the projections of the two paths sum in different orders, so h may differ in its last place
    err = (y.float() - ref.float()).abs()
    assert bool((err <= 2e-3 + 8e-3 * ref.float().abs()).all()), err.max().item()
    a, gate = h.chunk(2, dim=-1)
    ref32 = a.float() * F.gelu(gate.float())
    assert bool(((y.float() - ref32).abs() <= 2e-3 + 1.2e-2 * ref32.abs()).all())
    assert float((err == 0).float().mean()) > 0.95
    y2 = ops.linear_geglu(x, wp, bp)
    assert torch.equal(y, y2)                    # deterministic


def test_linear_geglu_rows_do_not_depend_on_m(cuda_device):
    """A row's result is the same whatever M is and whichever 256-row tile it lands in (no split-K): shard latents of
    a data-parallel run stay bit-identical to the single-GPU ones."""
    from photoverse_b200 import ops
    for C in (320, 640, 1280):
        x, w, b = _problem(cuda_device, 16384, C, C)
        wp, bp = ops.pack_geglu_weight(w, b)
        y = ops.linear_geglu(x, wp, bp)
        for r0, m in ((0, 32), (0, 2048), (1000, 512), (16384 - 200, 200)):
            assert torch.equal(ops.linear_geglu(x[r0:r0 + m].contiguous(), wp, bp), y[r0:r0 + m]), (C, r0, m)


def test_linear_geglu_packing_and_3d_input(cuda_device):
    """pack_geglu_weight's row order, and a [B, S, C] activation as the transformer blocks pass it."""
    from photoverse_b200 import ops
    x, w, b = _problem(cuda_device, 2 * 1024, 320, 9)
    wp, bp = ops.pack_geglu_weight(w, b)
    N = 1280
    j = torch.arange(N, device=w.device)
    assert torch.equal(wp[(j // 80) * 160 + j % 80], w[:N]) and torch.equal(wp[(j // 80) * 160 + 80 + j % 80], w[N:])
    assert torch.equal(bp[(j // 80) * 160 + 80 + j % 80], b[N:].float())
    y3 = ops.linear_geglu(x.view(2, 1024, 320), wp, bp)
    assert y3.shape == (2, 1024, N) and torch.equal(y3.view(-1, N), ops.linear_geglu(x, wp, bp))


def test_linear_geglu_rejects_malformed_arguments(cuda_device):
    from photoverse_b200 import _lib, ops
    x, w, b = _problem(cuda_device, 256, 320, 1)
    wp, bp = ops.pack_geglu_weight(w, b)
    with pytest.raises(_lib.PhotoverseB200Error, match="K %% 64|K % 64"):
        ops.linear_geglu(x[:, :160].contiguous(), wp[:, :160].contiguous(), bp)          # K = 160 fits no K-block count
    with pytest.raises(_lib.PhotoverseB200Error, match="N % 80"):
        ops.linear_geglu(x, wp[:200].contiguous(), bp[:200].contiguous())               # N = 100
    with pytest.raises(_lib.PhotoverseB200Error, match="features"):
        ops.linear_geglu(x[:, :256].contiguous(), wp, bp)
    with pytest.raises(_lib.PhotoverseB200Error, match="CUDA bfloat16"):
        ops.linear_geglu(x.float(), wp, bp)
    lib = _lib.lib()
    assert lib.pv_linear_geglu_fwd(1, None, None, None, None, 256, 1280, 320, 320, 1280, None) == 1
    assert b"null" in lib.pv_last_error()
    with pytest.raises(ValueError):
        ops.pack_geglu_weight(w[:200], b[:200])
