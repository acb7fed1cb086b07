"""What rtjgpu_decode_device_chw_window's binding decides without a device: the normalisation coefficients, and the
Python wrapper's dtype, order, coefficient and output checks (raised before anything reaches the library)."""
import numpy as np
import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D


def test_normalize_coefficients_imagenet():
    scale, bias = g.normalize_coefficients((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    assert scale.dtype == np.float32 and bias.dtype == np.float32 and scale.shape == bias.shape == (3,)
    # 1 / (255 std) and -mean / std, worked out in float64 and rounded once to float32
    want_scale = np.array([0.017124753831663668, 0.01750700280112045, 0.017429193899782137], np.float32)
    want_bias = np.array([-2.1179039301310043, -2.0357142857142856, -1.8044444444444445], np.float32)
    assert np.array_equal(scale.view(np.uint32), want_scale.view(np.uint32))
    assert np.array_equal(bias.view(np.uint32), want_bias.view(np.uint32))


def test_normalize_coefficients_rounds_once():
    """std = 1/255 gives scale 1 exactly; mean 0.5, std 0.5 gives 2/255 and -1."""
    scale, bias = capi.normalize_coefficients((0.0, 0.5, 1.0), (1 / 255, 0.5, 0.25))
    assert scale[0] == np.float32(1.0)
    assert scale[1] == np.float32(2.0 / 255.0) and bias[1] == np.float32(-1.0)
    assert scale[2] == np.float32(4.0 / 255.0) and bias[2] == np.float32(-4.0) and bias[0] == np.float32(-0.0)


@pytest.mark.parametrize("mean,std", [((0.5, 0.5), (0.5, 0.5, 0.5)), ((0.5, 0.5, 0.5), (0.5, 0.0, 0.5)),
                                      ((0.5, np.nan, 0.5), (0.5, 0.5, 0.5)), ((0.5, 0.5, 0.5), (0.5, np.inf, 0.5))])
def test_normalize_coefficients_refuses(mean, std):
    with pytest.raises(ValueError):
        capi.normalize_coefficients(mean, std)


def test_chw_constants_match_the_header():
    assert (capi.CHW_U8, capi.CHW_F16, capi.CHW_BF16, capi.CHW_F32) == (0, 1, 2, 3)
    assert capi.CHW_ESIZE == (1, 2, 2, 4)
    assert D.CHW_DTYPES == {torch.uint8: 0, torch.float16: 1, torch.bfloat16: 2, torch.float32: 3}
    assert D.CHW_ORDERS == {"rgb": capi.CONV_RGB24, "bgr": capi.CONV_BGR24}


class _Batch:
    """Enough of a DeviceBatch for arguments refused before it is looked at"""
    F, w, h, fmt = 4, 64, 48, 0


def _call(**kw):
    args = dict(dtype=torch.float16)
    args.update(kw)
    return D.decode_chw_window(None, _Batch(), [0, 2, 4], [0, 3], (32, 32), (0, 0), **args)


@pytest.mark.parametrize("kw", [
    dict(dtype=torch.int16), dict(dtype=torch.float64),                          # element types the call has not
    dict(order="rgba"), dict(order="RGB"),
    dict(mean=(0.5, 0.5, 0.5)), dict(std=(0.5, 0.5, 0.5)),                       # mean without std, and the converse
    dict(mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), scale=(1, 1, 1)),            # both ways of saying it
    dict(dtype=torch.uint8, scale=(1, 1, 1)), dict(dtype=torch.uint8, bias=(0, 0, 0)),
    dict(dtype=torch.uint8, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)),
    dict(mirror=[1, 0, 1]),                                                      # three flags for two sequences
    dict(out=torch.empty((2, 3, 32, 32), dtype=torch.float32)),                  # out of another dtype
    dict(out=torch.empty((2, 32, 32, 3), dtype=torch.float16)),                  # ... or shape
    dict(out=torch.empty((3, 3, 32, 32), dtype=torch.float16)),
    dict(out=torch.empty((2, 3, 32, 64), dtype=torch.float16)[..., :32]),        # ... or not contiguous
])
def test_wrapper_refuses(kw):
    with pytest.raises(ValueError):
        _call(**kw)


def test_float3_refuses_other_lengths():
    with pytest.raises(ValueError):
        capi._float3((1.0, 2.0))
    assert capi._float3(None) is None
    assert list(capi._float3(np.array([1, 2, 3]))) == [1.0, 2.0, 3.0]
