"""CPU: the compute-dtype rule under torch.autocast (DESIGN.md 4.9) and the argument checks of pv_convert_fwd.

Without a GPU ``torch.autocast("cuda")`` disables itself, so the rule is checked through the pure helper that takes the
autocast state as an argument."""
import pytest
import torch

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32


@pytest.mark.parametrize("tensor_dtype,grad,autocast,expected", [
    # autocast off: the tensor dtype, as without autocast support
    (F32, False, None, F32), (F32, True, None, F32), (BF16, True, None, BF16), (F16, False, None, F16),
    # 16-bit hidden states keep their own dtype under either autocast dtype, with or without grad
    (BF16, False, BF16, BF16), (BF16, True, F16, BF16), (F16, False, BF16, F16), (F16, True, F16, F16),
    (BF16, True, BF16, BF16), (F16, False, F16, F16),
    # float32 under bf16 autocast: bf16 in both modes
    (F32, False, BF16, BF16), (F32, True, BF16, BF16),
    # float32 under fp16 autocast: fp16 without grad; in grad mode float32 (there is no fp16 backward)
    (F32, False, F16, F16), (F32, True, F16, F32),
])
def test_compute_dtype_rule(tensor_dtype, grad, autocast, expected):
    from photoverse_b200 import ops
    assert ops.resolve_compute_dtype(tensor_dtype, grad, autocast) == expected


def test_compute_dtype_without_autocast_is_the_tensor_dtype():
    from photoverse_b200 import ops
    assert ops.autocast_dtype() is None
    for dt in (BF16, F16, F32):
        for grad in (False, True):
            assert ops.compute_dtype(dt, grad) == dt


@pytest.mark.parametrize("in_dt,out_dt", [(0, 0), (1, 1), (2, 2), (1, 2), (2, 1), (0, 7), (5, 0)])
def test_convert_rejects_unsupported_pairs_by_name(in_dt, out_dt):
    from photoverse_b200 import _lib
    lib = _lib.lib()
    assert lib.pv_convert_fwd(in_dt, out_dt, None, None, 8, None) == 3                 # PV_ERR_UNSUPPORTED
    msg = lib.pv_last_error().decode()
    names = {0: "PV_F32", 1: "PV_BF16", 2: "PV_F16"}
    assert "pv_convert_fwd" in msg
    for dt in (in_dt, out_dt):
        assert names.get(dt, "unknown pv_dtype") in msg, msg


@pytest.mark.parametrize("in_dt,out_dt", [(0, 1), (0, 2), (1, 0), (2, 0)])
def test_convert_rejects_bad_arguments_before_any_device_call(in_dt, out_dt):
    from photoverse_b200 import _lib
    lib = _lib.lib()
    assert lib.pv_convert_fwd(in_dt, out_dt, None, None, -1, None) == 1                # PV_ERR_INVALID
    assert "n must be >= 0" in lib.pv_last_error().decode()
    assert lib.pv_convert_fwd(in_dt, out_dt, None, None, 8, None) == 1
    assert "null pointer" in lib.pv_last_error().decode()
    assert lib.pv_convert_fwd(in_dt, out_dt, 4097, 8192, 8, None) == 1                  # odd address: not element-aligned
    assert "aligned" in lib.pv_last_error().decode()
    n0 = lib.pv_launch_count()
    assert lib.pv_convert_fwd(in_dt, out_dt, None, None, 0, None) == 0                 # nothing to convert, nothing launched
    assert lib.pv_launch_count() == n0


def test_ops_convert_refuses_cpu_tensors():
    from photoverse_b200 import _lib, ops
    with pytest.raises(_lib.PhotoverseB200Error, match="CUDA"):
        ops.convert(torch.zeros(8), torch.bfloat16)


def test_trainer_refuses_fp16_autocast():
    from photoverse_b200.host.train_step import Trainer
    with pytest.raises(ValueError, match="float16"):
        Trainer(None, None, None, autocast_dtype=torch.float16)
