"""CPU: float16 is a compute dtype of the inference entry points only.  Every other entry point of the C ABI rejects
PV_F16 by name, before it looks at its arguments, and the Python front end maps torch.float16 to it."""
import pytest
import torch


def test_pv_f16_value_and_dtype_mapping():
    from photoverse_b200 import _lib, ops
    assert (_lib.PV_F32, _lib.PV_BF16, _lib.PV_F16) == (0, 1, 2)
    assert ops._code(torch.float16) == _lib.PV_F16 and ops._code(torch.bfloat16) == _lib.PV_BF16
    with pytest.raises(_lib.PhotoverseB200Error, match="bfloat16, float16 .*float32"):
        ops._code(torch.float64)


@pytest.mark.parametrize("name,args", [
    ("pv_pack_weight_t", [None, None, None, 0.0, None, 8, 8, 0, None]),
    ("pv_transpose_2d", [None, None, 8, 8, 8, 8, None]),
    ("pv_linear_bwd_weight", [None, None, None, None, 8, 8, 8, 8, 8, 1.0, 0.0, None]),
    ("pv_lora_bwd", [None, None, None, None, 1.0, None, None, 8, 8, 8, 1, 8, 8, None]),
    ("pv_col_sum", [None, None, None, 8, 8, 8, None]),
    ("pv_ln_lrelu_bwd", [None] * 10 + [1, 1, 1024, 0.01, None]),
    ("pv_group_mean_bwd", [None, None, 1, 1, 8, 8, None]),
    ("pv_dual_attn_bwd", [None] * 7 + [1, 256, 320, 8, 77, 1, 1.0, 1.0, None]),
    ("pv_kv_pack_bwd", [None] * 6 + [1, 256, 77, 1, 320, 8, None]),
    ("pv_inject_concept_fwd", [None, None, None, None, 1, 77, 1, 768, None]),
    ("pv_train_loss_fwd", [None, None, 8, None, 0, None, 0, 0.01, 0.001, None, None, None]),
    ("pv_dropout_bwd_acc", [None, None, None, 1.0, 8, None]),
    ("pv_group_norm_nhwc_fwd", [None] * 7 + [1, 64, 320, 32, 1e-5, 1, None]),
    ("pv_layer_norm_fwd", [None] * 6 + [8, 320, 1e-5, None]),
    ("pv_geglu_fwd", [None, None, 8, 80, 160, None]),
    ("pv_linear_geglu_fwd", [None, None, None, None, 8, 80, 64, 64, 80, None]),
])
def test_entry_points_outside_the_inference_path_reject_f16(name, args):
    from photoverse_b200 import _lib
    lib = _lib.lib()
    assert getattr(lib, name)(_lib.PV_F16, *args) == 3                  # PV_ERR_UNSUPPORTED
    msg = lib.pv_last_error().decode()
    assert name in msg and "PV_F16" in msg, msg


def test_wgrad_workspace_query_rejects_f16():
    from photoverse_b200 import _lib
    lib = _lib.lib()
    assert lib.pv_linear_bwd_weight_ws_bytes(_lib.PV_F16, 512, 128, 128) == -1
    assert "PV_F16" in lib.pv_last_error().decode()


def test_kv_tile_bytes_f16_equals_bf16():
    from photoverse_b200 import _lib
    lib = _lib.lib()
    for C in (320, 640, 1280):
        assert lib.pv_kv_tile_bytes(_lib.PV_F16, C, 8, 77, 5) == lib.pv_kv_tile_bytes(_lib.PV_BF16, C, 8, 77, 5) > 0
