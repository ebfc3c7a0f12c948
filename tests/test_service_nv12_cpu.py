"""The service's out_fmt keyword without a GPU: which formats the constructor takes, and the frame shapes NV12 output has
(including the frame-less entries the temporal delay line returns while it fills)."""
import pytest
import torch

from ss4k_b200 import _lib as L
from ss4k_b200 import service


@pytest.mark.parametrize("out_fmt", [L.FMT_U8_NHWC, L.FMT_NV12])
def test_constructor_accepts_rgb_and_nv12_without_a_device(out_fmt):
    svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, out_fmt=out_fmt)
    assert svc.out_fmt == out_fmt and svc.model is None


def test_constructor_default_is_uint8_rgb():
    assert service.FsrcnnUpscalerService(device=0).out_fmt == L.FMT_U8_NHWC


@pytest.mark.parametrize("out_fmt", [L.FMT_F32_NCHW, L.FMT_F16_NCHW, 4, -1, "nv12", None])
def test_constructor_rejects_other_formats(out_fmt):
    with pytest.raises(ValueError):
        service.FsrcnnUpscalerService(device=0, out_fmt=out_fmt)


def test_frame_shape():
    assert service.frame_shape(L.FMT_U8_NHWC, 1440, 2560) == (1440, 2560, 3)
    assert service.frame_shape(L.FMT_NV12, 1440, 2560) == (2160, 2560)
    assert service.frame_shape(L.FMT_NV12, 180, 320) == (270, 320)
    assert service.frame_shape(L.FMT_NV12, 0, 0) == (0, 0)
    assert service.frame_shape(L.FMT_U8_NHWC, 181, 322) == (181, 322, 3)   # any size in RGB


@pytest.mark.parametrize("h,w", [(181, 320), (180, 322), (180, 321), (1, 4)])
def test_frame_shape_refuses_sizes_nv12_cannot_hold(h, w):
    with pytest.raises(L.Ss4kError, match="NV12"):
        service.frame_shape(L.FMT_NV12, h, w)


def test_frame_shape_rejects_other_formats():
    with pytest.raises(ValueError):
        service.frame_shape(L.FMT_F16_NCHW, 16, 16)


@pytest.mark.parametrize("out_fmt,output_shape,want", [
    (L.FMT_U8_NHWC, None, (0, 0, 0, 3)),
    (L.FMT_U8_NHWC, (1440, 2560), (0, 1440, 2560, 3)),
    (L.FMT_NV12, None, (0, 0, 0)),
    (L.FMT_NV12, (1440, 2560), (0, 2160, 2560)),
])
def test_frame_less_entries(out_fmt, output_shape, want):
    svc = service.FsrcnnUpscalerService(device=torch.device("cpu"), out_fmt=out_fmt)
    svc.output_shape = output_shape
    got = svc._no_frames()
    assert tuple(got.shape) == want and got.dtype == torch.uint8
