"""CPU-side checks of the bf16 crop-layer entry points: argument validation happens before any CUDA call (so it is testable
without a GPU), the messages name the function called, and the Python wrapper rejects CPU tensors and unsupported dtypes."""
import ctypes

import pytest
import torch

from hands_b200 import _lib

P = ctypes.c_void_p


def _msg(lib):
    return lib.hb_last_error_string().decode()


def test_bf16_forward_argument_errors():
    lib = _lib.load()
    d = P(256)   # never dereferenced: every call below fails validation first
    mean = (ctypes.c_float * 3)(0.5, 0.5, 0.5)
    std = (ctypes.c_float * 3)(0.25, 0.25, 0.25)
    m, s = ctypes.cast(mean, P), ctypes.cast(std, P)
    # NULL pointers
    assert lib.hb_pcl_fwd_bf16(None, None, 3, 1, 3, 224, None, None) == -1 and "hb_pcl_fwd_bf16" in _msg(lib)
    assert lib.hb_pcl_fwd_bf16(d, d, 2, 1, 3, 224, None, None) == -1
    assert lib.hb_pcl_fwd_u8_bf16(d, m, s, d, 2, 1, 3, 224, None, None) == -1 and "hb_pcl_fwd_u8_bf16" in _msg(lib)
    assert lib.hb_pcl_fwd_u8_bf16(d, None, s, d, 2, 1, 3, 224, d, None) == -1 and "hb_pcl_fwd_u8_bf16" in _msg(lib)
    # C out of range
    for C in (0, 5):
        assert lib.hb_pcl_fwd_bf16(d, d, 2, 1, C, 224, d, None) == -1 and "hb_pcl_fwd_bf16" in _msg(lib)
        assert lib.hb_pcl_fwd_u8_bf16(d, m, s, d, 2, 1, C, 224, d, None) == -1 and "hb_pcl_fwd_u8_bf16" in _msg(lib)
    # n_crops not a multiple of crops_per_img, and crops_per_img <= 0
    assert lib.hb_pcl_fwd_bf16(d, d, 3, 2, 3, 224, d, None) == -1
    assert lib.hb_pcl_fwd_bf16(d, d, 2, 0, 3, 224, d, None) == -1
    assert lib.hb_pcl_fwd_u8_bf16(d, m, s, d, 3, 2, 3, 224, d, None) == -1 and "hb_pcl_fwd_u8_bf16" in _msg(lib)
    # a zero std
    std0 = (ctypes.c_float * 3)(0.25, 0.0, 0.25)
    assert lib.hb_pcl_fwd_u8_bf16(d, m, ctypes.cast(std0, P), d, 2, 1, 3, 224, d, None) == -1 and "std[1]" in _msg(lib)
    # an empty batch is a no-op, as for the fp32 twins
    assert lib.hb_pcl_fwd_bf16(None, None, 0, 1, 3, 224, None, None) == 0
    assert lib.hb_pcl_fwd_u8_bf16(None, m, s, None, 0, 1, 3, 224, None, None) == 0


def test_bf16_backward_argument_errors():
    lib = _lib.load()
    d = P(256)
    one_img = lib.hb_pcl_bwd_workspace_bytes(2, 2, 3, 224)   # one image of two crops
    assert one_img == 2 * 4 * 224 * 224 * 4
    # NULL pointers, C out of range, n_crops % crops_per_img
    assert lib.hb_pcl_bwd_bf16(None, d, 2, 2, 3, 224, d, d, one_img, None) == -1 and "hb_pcl_bwd_bf16" in _msg(lib)
    assert lib.hb_pcl_bwd_bf16(d, d, 2, 2, 3, 224, d, None, one_img, None) == -1
    assert lib.hb_pcl_bwd_bf16(d, d, 2, 2, 0, 224, d, d, one_img, None) == -1 and "hb_pcl_bwd_bf16" in _msg(lib)
    assert lib.hb_pcl_bwd_bf16(d, d, 2, 2, 5, 224, d, d, one_img, None) == -1
    assert lib.hb_pcl_bwd_bf16(d, d, 3, 2, 3, 224, d, d, one_img, None) == -1
    # a workspace smaller than one image's worth
    rc = lib.hb_pcl_bwd_bf16(d, d, 4, 2, 3, 224, d, d, one_img - 16, None)
    assert rc == -3 and "hb_pcl_bwd_bf16" in _msg(lib) and "workspace too small" in _msg(lib)
    # the fp32 twin keeps its own messages
    assert lib.hb_pcl_bwd(d, d, 4, 2, 3, 224, d, d, one_img - 16, None) == -3 and _msg(lib).startswith("hb_pcl_bwd:")
    assert lib.hb_pcl_bwd_bf16(None, None, 0, 2, 3, 224, None, None, 0, None) == 0


def test_perspective_crop_out_dtype_on_cpu():
    from hands_b200.pcl import perspective_crop

    bbox = torch.tensor([[10, 10, 100, 90]], dtype=torch.int32)
    K = torch.tensor([[[500.0, 0, 112], [0, 500.0, 112], [0, 0, 1]]])
    with pytest.raises(RuntimeError, match="no CPU path"):
        perspective_crop(torch.zeros(1, 3, 224, 224), bbox, K, out_dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        perspective_crop(torch.zeros(1, 3, 224, 224, dtype=torch.uint8), bbox, K, mean=(0.5,) * 3, std=(0.2,) * 3, out_dtype=torch.bfloat16)
    for bad in (torch.float16, torch.float64, torch.uint8, "bf16"):
        with pytest.raises(TypeError, match="out_dtype"):
            perspective_crop(torch.zeros(1, 3, 224, 224), bbox, K, out_dtype=bad)


def test_geometry_step_rejects_bad_crop_dtype():
    from hands_b200.step import GeometryStep

    with pytest.raises(TypeError, match="out_dtype"):
        GeometryStep(2, "cpu", crop_dtype=torch.float16)
