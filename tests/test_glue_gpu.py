"""The service glue kernels (csrc/glue.cu), one C entry at a time, against plain float64 references of the same operation
computed on the CPU from the very values the kernel reads (uint8 as float32(v / 255), half widened exactly), and the
whole glue as the service drives it against the uint8 outputs of the reference's own code (tests/golden/glue.npz).

The whole-service tests (test_service_gpu.py, test_cfg3_gpu.py) put a network in front of the glue, so their tolerances
absorb the nets' fp16 error; a glue defect smaller than that passes there.  Here the tolerances are those of one fp32
evaluation, so a wrong coefficient, index or rounding mode shows.

Tolerance rules (one place, argued once):
  * float outputs: a sum of k fp32 products is within about k * u * sum|terms| of the exact value (u = 2^-24); the
    entries evaluate at most ~16 terms per output, so |got - ref| <= 1e-6 * sum|terms| (16 u = 9.5e-7), except the
    289-tap blur (1e-5) and area pooling (window size + 1) * u.
  * 16-bit outputs: the fp32 value (within 2e-6 of the exact one for these O(1) sums) rounded to nearest, so within
    half an ulp of the 16-bit type of the fp64 value plus 2e-6.
  * uint8 outputs: the kernel's float is within ~1e-6 * sum|terms| (a few 1e-6 with the coordinate rounding of the
    resamplers on smooth images) of the fp64 value, i.e. under EPS_U8 = 2e-3 on the x255 scale.  So the byte equals
    floor (rint with round_u8) of 255 * ref, and may differ by one level only where 255 * ref lies within EPS_U8 of the
    rounding boundary.
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from ss4k_b200 import _lib as L
from ss4k_b200 import service
from oracle import colour, glue, srvgg

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
E_INVALID = -1   # SS4K_E_INVALID
EPS_U8 = 2e-3
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---------------------------------------------------------------- calling the C entries
def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _call(engine, name, *args):
    """engine.lib.<name>(*args, current stream) as service.py calls it; returns the status after the work finished."""
    rc = getattr(engine.lib, name)(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc


def _ok(engine, name, *args):
    rc = _call(engine, name, *args)
    assert rc == L.OK, (name, rc)


def _at_offset(t, offset, pad=0):
    """A copy of device tensor ``t`` as a view ``offset`` elements into a larger allocation (``pad`` more behind)."""
    buf = torch.zeros(t.numel() + offset + pad, dtype=t.dtype, device=t.device)
    v = buf[offset:offset + t.numel()].view(t.shape)
    v.copy_(t)
    return v


# ---------------------------------------------------------------- inputs
def _smooth(n, c, h, w, seed, lo=0.0, hi=1.0):
    """fp64 NCHW image: a random image at ~1/8 resolution, bilinearly enlarged (slope below 1/8 per pixel, so the
    resamplers' float32 coordinate rounding stays far below EPS_U8), plus fine noise."""
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(n, c, h // 8 + 2, w // 8 + 2, generator=g, dtype=torch.float64)
    v = F.interpolate(base, size=(h, w), mode="bilinear", align_corners=False)
    v = v + 0.01 * torch.rand(n, c, h, w, generator=g, dtype=torch.float64)
    return lo + (hi - lo) * (v - v.min()) / (v.max() - v.min())


def _noise(n, c, h, w, seed, lo=0.0, hi=1.0):
    g = torch.Generator().manual_seed(seed)
    return lo + (hi - lo) * torch.rand(n, c, h, w, generator=g, dtype=torch.float64)


def _as_fmt(v, fmt):
    """fp64 NCHW values -> (device tensor in glue format fmt: 0 float NCHW, 1 half NCHW, 2 uint8 NHWC;
    fp64 NCHW of exactly the values the kernels read)."""
    if fmt == 2:
        u8 = (v.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        return u8.cuda(), (u8.permute(0, 3, 1, 2).float() / 255.0).double()
    t = v.half() if fmt == 1 else v.float()
    return t.cuda(), t.double()


def _nv12(n, h, w, seed):
    """Random NV12 frames (uint8 [n, h*w*3/2]) and their RGB decode by the colour oracle (fp64 NCHW)."""
    g = torch.Generator().manual_seed(seed)
    nv = torch.randint(16, 236, (n, h * w * 3 // 2), dtype=torch.uint8, generator=g)
    return nv.cuda(), torch.from_numpy(colour.nv12_to_rgb(nv.numpy(), h, w)).double()


def _other(fmt, n, c, h, w, seed):
    if fmt is None:
        return None, None
    if fmt == 3:
        return _nv12(n, h, w, seed)
    return _as_fmt(_noise(n, c, h, w, seed), fmt)


# ---------------------------------------------------------------- tolerance helpers
def _assert_f32(got, ref, mag, rel, what, slack=0.0):
    """|got - ref| <= rel * mag + slack elementwise, mag = sum of |terms| of each output (see the module docstring)."""
    err = (got.double().cpu() - ref).abs()
    bound = rel * mag + slack
    worst = (err / bound.clamp_min(1e-300)).max().item()
    print(f"{what}: max |err| {err.max().item():.3e}, worst err / bound {worst:.3f}")
    assert (err <= bound).all(), (what, worst)


def _assert_16(got, ref, bf16, what):
    """got: 16-bit tensor (half or bfloat16); within half an ulp (of the larger of |got|, |ref|) of ref, plus 2e-6."""
    mant, emin = (7, -126) if bf16 else (10, -14)
    g = got.double().cpu()
    m = torch.maximum(g.abs(), ref.abs()).clamp_min(2.0 ** emin)
    ulp = torch.pow(2.0, torch.floor(torch.log2(m)) - mant)
    err = (g - ref).abs()
    worst = (err / (0.5 * ulp + 2e-6)).max().item()
    print(f"{what}: max |err| {err.max().item():.3e}, worst err / bound {worst:.3f}")
    assert (err <= 0.5 * ulp + 2e-6).all(), (what, worst)


def _assert_u8(got, ref255, round_u8, what):
    """got: uint8; ref255: 255 * the fp64 value (clamped), same layout.  Exact floor / rint, one level of slack only
    within EPS_U8 of the boundary."""
    ref255 = ref255.double().cpu()
    want = torch.round(ref255) if round_u8 else torch.floor(ref255)      # rintf and torch.round: half to even
    frac = ref255 - torch.floor(ref255)
    dist = (frac - 0.5).abs() if round_u8 else torch.minimum(frac, 1.0 - frac)
    d = got.cpu().double() - want
    flip = d != 0
    far = dist[flip].max().item() if flip.any() else 0.0
    print(f"{what}: {int(flip.sum())} of {d.numel()} values one level off, largest boundary distance of a flip {far:.2e}")
    assert d.abs().max().item() <= 1, what
    assert far <= EPS_U8, (what, far)


# ---------------------------------------------------------------- fp64 references
def _stats64(v):
    n, c = v.shape[:2]
    x = v.reshape(n, c, -1)
    return x.sum(-1), (x * x).sum(-1)


def _match64(hr, lr):
    """match_mean_std's affine map (fsrcnn_upscaler.py:188-199): a = std_lr / (std_hr + 1e-8), b = mean_lr - a * mean_hr,
    unbiased std; shapes [n, c, 1, 1]."""
    n, c = hr.shape[:2]
    hs, ls = hr.reshape(n, c, -1).std(-1), lr.reshape(n, c, -1).std(-1)
    a = ls / (hs + 1e-8)
    b = lr.reshape(n, c, -1).mean(-1) - a * hr.reshape(n, c, -1).mean(-1)
    return a.view(n, c, 1, 1), b.view(n, c, 1, 1)


def _sharpen64(x, strength, opacity, other):
    """opacity * clamp(sharpen_ker(strength)(x), 0, 1) + (1 - opacity) * other, sum|terms|  (fsrcnn_upscaler.py:278-281)."""
    n, c, h, w = x.shape
    k = glue.sharpen_weight(strength).double()
    conv = lambda t, kk: glue.depthwise_reflect(t.reshape(n * c, 1, h, w), kk).reshape(n, c, h, w)  # noqa: E731
    v = conv(x, k).clamp(0, 1)
    mag = conv(x.abs(), k.abs())
    if other is not None:
        v = opacity * v + (1 - opacity) * other
        mag = opacity * mag + (1 - opacity) * other.abs()
    return v, mag


def _stats_dev(engine, img, fmt, n, c, h, w):
    sums = torch.empty(n * c, 2, dtype=torch.float64, device="cuda")
    _ok(engine, "ss4k_glue_chan_stats", _p(img), fmt, n, c, h, w, _p(sums))
    return sums


def _match_inputs(n, c, h, w, lh, lw, seed):
    """An HR image (half) and a small LR image (float) with per-image different distributions, their engine statistics
    and the fp64 affine map.  The LR image is small so that the unbiased / biased variance ratio is far from 1."""
    scale = torch.linspace(0.5, 1.0, n, dtype=torch.float64).view(n, 1, 1, 1)
    hr_dev, hr64 = _as_fmt(_smooth(n, c, h, w, seed) * scale + 0.05, 1)
    lr_dev, lr64 = _as_fmt(_noise(n, c, lh, lw, seed + 1, 0.2, 0.8), 0)
    return hr_dev, hr64, lr_dev, lr64


# ---------------------------------------------------------------- chan_stats
@pytest.mark.parametrize("fmt,n,c,h,w,offset", [
    (1, 1, 3, 1440, 2560, 0),   # half, vectorised kernel, one 4x-frame plane (grid-stride)
    (1, 2, 3, 64, 96, 0),       # half, vectorised kernel
    (1, 3, 4, 30, 35, 0),       # half, h*w % 8 != 0: general kernel; n*c = 12
    (1, 2, 3, 64, 96, 1),       # half view at an odd element offset: general kernel
    (0, 4, 3, 37, 41, 0),
    (0, 1, 3, 2, 3, 0),         # tiny plane
    (2, 2, 3, 45, 80, 0),
    (2, 1, 1, 2, 3, 0),
])
def test_chan_stats(engine, fmt, n, c, h, w, offset):
    dev, v64 = _as_fmt(_noise(n, c, h, w, 1, -0.5, 1.5) if fmt != 2 else _noise(n, c, h, w, 1), fmt)
    if offset:
        dev = _at_offset(dev, offset)
    s, q = _stats64(v64)
    sums = torch.full((n * c, 2), float("nan"), dtype=torch.float64, device="cuda")
    for _ in range(2):   # twice into the same buffer: the entry zeroes it first
        _ok(engine, "ss4k_glue_chan_stats", _p(dev), fmt, n, c, h, w, _p(sums))
        got = sums.cpu().view(n, c, 2)
        # double accumulation of exactly representable values: only the summation order differs
        assert ((got[..., 0] - s).abs() <= 1e-12 * v64.abs().reshape(n, c, -1).sum(-1)).all()
        assert ((got[..., 1] - q).abs() <= 1e-12 * q).all()


# ---------------------------------------------------------------- area_pool
@pytest.mark.parametrize("fmt,n,c,h,w,oh,ow", [
    (0, 2, 3, 64, 96, 32, 48),          # factor 2
    (1, 2, 3, 96, 128, 12, 16),         # factor 8: the colour match's pooling
    (2, 1, 3, 1080, 1920, 720, 1280),   # 1.5: the LR area downscale
    (0, 1, 3, 97, 131, 13, 17),         # ragged windows
    (1, 2, 3, 20, 30, 20, 30),          # identity
    (2, 1, 3, 10, 14, 25, 33),          # up-pooling
    (0, 2, 3, 37, 53, 1, 1),            # one output pixel
])
def test_area_pool(engine, fmt, n, c, h, w, oh, ow):
    dev, v64 = _as_fmt(_noise(n, c, h, w, 2), fmt)
    out = torch.full((n, c, oh, ow), float("nan"), dtype=torch.float32, device="cuda")
    _ok(engine, "ss4k_glue_area_pool", _p(dev), fmt, n, c, h, w, _p(out), oh, ow)
    ref = F.adaptive_avg_pool2d(v64, (oh, ow))
    k = (-(-h // oh) + 1) * (-(-w // ow) + 1)   # largest window: k fp32 additions and a division
    _assert_f32(out, ref, F.adaptive_avg_pool2d(v64.abs(), (oh, ow)), (k + 1) * U32 * 1.01, "area_pool")


# ---------------------------------------------------------------- blur_diff
@pytest.mark.parametrize("ksize,n,c,h,w,with_sums", [
    (17, 2, 3, 12, 16, True),    # the service's gaussian_kernel(17, 8.0) on a 96 x 128 frame's 1/8 image
    (17, 1, 3, 9, 9, False),     # h = w = ksize // 2 + 1: the reflect limit
    (17, 2, 3, 9, 23, True),
    (17, 1, 3, 31, 9, True),
    (3, 2, 3, 2, 7, True),
    (5, 1, 3, 13, 3, False),
    (5, 2, 3, 11, 14, True),
])
def test_blur_diff(engine, ksize, n, c, h, w, with_sums):
    kern = service.gaussian_kernel(17, 8.0) if ksize == 17 else glue.blur_weight(ksize, 0.3 * ksize)[0, 0]
    hb_dev, hb = _as_fmt(_noise(n, c, h, w, 3, 0.1, 0.9), 0)
    lb_dev, lb = _as_fmt(_noise(n, c, h, w, 4, 0.1, 0.9), 0)
    a, b = torch.ones(n, c, 1, 1, dtype=torch.float64), torch.zeros(n, c, 1, 1, dtype=torch.float64)
    hs = ls = None
    cnt_hr = cnt_lr = 0.0
    if with_sums:   # statistics of the full-size images the engine's own chan_stats produced
        hr_dev, hr64, lr_dev, lr64 = _match_inputs(n, c, 8 * h, 8 * w, 6, 10, 5)
        hs = _stats_dev(engine, hr_dev, 1, n, c, 8 * h, 8 * w)
        ls = _stats_dev(engine, lr_dev, 0, n, c, 6, 10)
        cnt_hr, cnt_lr = float(64 * h * w), 60.0
        a, b = _match64(hr64, lr64)
    diff = torch.full((n, c, h, w), float("nan"), dtype=torch.float32, device="cuda")
    _ok(engine, "ss4k_glue_blur_diff", _p(hb_dev), _p(lb_dev), _p(diff), _p(kern.cuda()), ksize, n, c, h, w, _p(hs), _p(ls),
        cnt_hr, cnt_lr)
    k64 = kern.double().view(1, 1, ksize, ksize)
    conv = lambda t: glue.depthwise_reflect(t.reshape(n * c, 1, h, w), k64).reshape(n, c, h, w)  # noqa: E731
    ref = conv(a * hb + b - lb)
    mag = conv((a * hb).abs() + b.abs() + lb.abs())
    _assert_f32(diff, ref, mag, 1e-5, f"blur_diff k{ksize}")


# ---------------------------------------------------------------- finalize
def _finalize64(hr64, a, b, diff64):
    """clamp(a*hr + b - bilinear_up(diff), 0, 1), sum|terms|, and the absolute slack of the kernel's float32 source
    coordinates: off by ~2u * coordinate, times the slope of diff (below 2 max|diff| per cell)  (fsrcnn_upscaler.py:
    197-198,214-220)."""
    h, w = hr64.shape[-2:]
    v, mag, slack = a * hr64 + b, (a * hr64).abs() + b.abs(), 0.0
    if diff64 is not None:
        up = F.interpolate(diff64, size=(h, w), mode="bilinear", align_corners=False)
        v, mag = v - up, mag + F.interpolate(diff64.abs(), size=(h, w), mode="bilinear", align_corners=False)
        dh, dw = diff64.shape[-2:]
        slack = 4.0 * U32 * (dh + dw) * diff64.abs().max().item()
    return v.clamp(0, 1), mag, slack


def _diff_shape(mode, h, w):
    return {None: None, "1/8": (max(h // 8, 1), max(w // 8, 1)), "1/2": (h // 2, w // 2), "full": (h, w)}[mode]


def _diff(n, c, shape, seed):
    if shape is None:
        return None, None
    d = _smooth(n, c, *shape, seed, -0.15, 0.15)
    return d.float().cuda(), d.float().double()


@pytest.mark.parametrize("fmt,n,c,h,w,dmode,out,round_u8,sums", [
    (1, 3, 3, 15, 17, None, "u8", 0, True),       # plane 255 < 256: per-pixel coefficients
    (0, 3, 3, 16, 16, "full", "u8", 1, True),     # plane 256: blocks aligned to images
    (1, 3, 3, 1, 257, "full", "f32", 0, True),    # plane 257: blocks straddle two images
    (1, 3, 3, 1, 257, None, "u8", 0, True),
    (1, 2, 3, 64, 96, "1/8", "u8", 0, True),      # the service's shape of the call
    (0, 2, 3, 72, 100, "1/8", "f32", 0, True),
    (1, 2, 3, 72, 100, "1/8", "u8", 1, False),    # NULL sums: a = 1, b = 0
    (1, 2, 1, 20, 30, "full", "u8", 0, True),     # C = 1: per-pixel coefficients, byte stores
    (0, 2, 1, 20, 30, "1/8", "f32", 0, True),
    (0, 2, 5, 24, 40, "1/8", "f32", 0, True),     # C = 5: per-pixel coefficients
    (1, 3, 3, 13, 29, "1/8", "u8", 0, True),      # 1131 pixels: ragged last warp
])
def test_finalize(engine, fmt, n, c, h, w, dmode, out, round_u8, sums):
    hr_dev, hr64, lr_dev, lr64 = _match_inputs(n, c, h, w, 6, 8, 7)
    if fmt == 0:
        hr_dev = hr_dev.float()
    hs = ls = None
    a, b = torch.ones(n, c, 1, 1, dtype=torch.float64), torch.zeros(n, c, 1, 1, dtype=torch.float64)
    if sums:
        hs, ls = _stats_dev(engine, hr_dev, fmt, n, c, h, w), _stats_dev(engine, lr_dev, 0, n, c, 6, 8)
        a, b = _match64(hr64, lr64)
    dshape = _diff_shape(dmode, h, w)
    d_dev, d64 = _diff(n, c, dshape, 8)
    dh, dw = dshape if dshape else (0, 0)
    ref, mag, slack = _finalize64(hr64, a, b, d64)
    args = (_p(hr_dev), fmt, n, c, h, w, _p(d_dev), dh, dw, _p(hs), _p(ls), float(h * w), 48.0)
    if out == "f32":
        got = torch.full((n, c, h, w), float("nan"), dtype=torch.float32, device="cuda")
        _ok(engine, "ss4k_glue_finalize", *args, None, _p(got), round_u8)
        _assert_f32(got, ref, mag, 1e-6, "finalize f32", slack)
        return
    got = torch.full((n, h, w, c), 7, dtype=torch.uint8, device="cuda")
    _ok(engine, "ss4k_glue_finalize", *args, _p(got), None, round_u8)
    _assert_u8(got, (ref * 255).permute(0, 2, 3, 1), round_u8, "finalize u8")
    # the same into a view at byte offset 1: unpacked byte stores, same bytes
    odd = _at_offset(torch.full_like(got, 9), 1, pad=3)
    _ok(engine, "ss4k_glue_finalize", *args, _p(odd), None, round_u8)
    assert torch.equal(odd, got)


# ---------------------------------------------------------------- bicubic_u8
def _bicubic255(v64, oh, ow):
    """F.interpolate(mode='bicubic', align_corners=False) (A = -0.75, border-replicated taps), clamp, x255, NHWC."""
    return (F.interpolate(v64, size=(oh, ow), mode="bicubic", align_corners=False).clamp(0, 1) * 255).permute(0, 2, 3, 1)


@pytest.mark.parametrize("n,c,h,w,oh,ow,round_u8", [
    (2, 3, 40, 56, 100, 140, 0),   # up 2.5
    (1, 3, 100, 140, 40, 56, 0),   # down 2.5
    (1, 1, 30, 50, 97, 131, 1),    # C = 1, non-integer up
    (2, 3, 90, 160, 31, 45, 0),    # down ~3.5
    (1, 3, 17, 23, 1, 1, 0),       # one output pixel
    (1, 1, 64, 64, 150, 40, 1),    # up along y, down along x
])
def test_bicubic_u8(engine, n, c, h, w, oh, ow, round_u8):
    v64 = _smooth(n, c, h, w, 9, -0.05, 1.05).float().double()
    out = torch.full((n, oh, ow, c), 7, dtype=torch.uint8, device="cuda")
    _ok(engine, "ss4k_glue_bicubic_u8", _p(v64.float().cuda()), n, c, h, w, _p(out), oh, ow, round_u8)
    _assert_u8(out, _bicubic255(v64, oh, ow), round_u8, "bicubic_u8")


# ---------------------------------------------------------------- finalize_bicubic_u8
def _staged_tiles(h, oh, dh):
    """Which 8-row tiles of finalize_bicubic_u8_kernel stage their diff rows in shared memory (at most 6 rows touched),
    by the kernel's float32 arithmetic: returns (some tile staged, some tile not)."""
    fy = np.float32(h) / np.float32(oh)
    ry = np.float32(dh) / np.float32(h)
    staged = []
    for oy0 in range(0, oh, 8):
        oy1 = min(oy0 + 8, oh) - 1
        p0 = int(np.floor(np.float32(oy0 + 0.5) * fy - np.float32(0.5))) - 1
        p1 = int(np.floor(np.float32(oy1 + 0.5) * fy - np.float32(0.5))) + 2
        s0 = max(np.float32(min(max(p0, 0), h - 1) + 0.5) * ry - np.float32(0.5), 0.0)
        s1 = max(np.float32(min(max(p1, 0), h - 1) + 0.5) * ry - np.float32(0.5), 0.0)
        hi = int(s1) + 1 if int(s1) < dh - 1 else int(s1)
        staged.append(hi - int(s0) + 1 <= 6)
    return any(staged), not all(staged)


@pytest.mark.parametrize("fmt,n,h,w,oh,ow,dmode,round_u8", [
    (1, 2, 96, 128, 100, 140, "1/8", 0),   # the golden cases' resize: staged diff rows
    (1, 1, 160, 240, 80, 120, "1/8", 0),   # downscale exactly 2, staged
    (0, 2, 96, 128, 48, 64, "1/2", 0),     # diff at H/2: un-staged fallback
    (1, 1, 64, 96, 100, 150, "full", 1),   # diff at H: un-staged fallback
    (1, 1, 270, 200, 100, 99, "1/8", 0),   # fy = 2.7, just inside the guard; OW % 32, OH % 8, OW*3 % 4 != 0
    (0, 1, 50, 70, 37, 45, None, 0),       # no diff; no packed stores
    (1, 2, 72, 136, 144, 272, None, 1),
])
def test_finalize_bicubic_u8(engine, fmt, n, h, w, oh, ow, dmode, round_u8):
    c = 3
    hr_dev, hr64, lr_dev, lr64 = _match_inputs(n, c, h, w, 6, 8, 11)
    if fmt == 0:
        hr_dev = hr_dev.float()
    hs, ls = _stats_dev(engine, hr_dev, fmt, n, c, h, w), _stats_dev(engine, lr_dev, 0, n, c, 6, 8)
    a, b = _match64(hr64, lr64)
    dshape = _diff_shape(dmode, h, w)
    d_dev, d64 = _diff(n, c, dshape, 12)
    dh, dw = dshape if dshape else (0, 0)
    if dshape is not None:
        some_staged, some_not = _staged_tiles(h, oh, dh)
        assert (some_staged and not some_not) if dmode == "1/8" else some_not
    args = (_p(hr_dev), fmt, n, c, h, w, _p(d_dev), dh, dw, _p(hs), _p(ls), float(h * w), 48.0)
    fused = torch.full((n, oh, ow, c), 7, dtype=torch.uint8, device="cuda")
    _ok(engine, "ss4k_glue_finalize_bicubic_u8", *args, _p(fused), oh, ow, round_u8)
    ref = _finalize64(hr64, a, b, d64)[0]
    _assert_u8(fused, _bicubic255(ref, oh, ow), round_u8, "finalize_bicubic_u8")
    # the same arithmetic as finalize (float NCHW) followed by bicubic_u8: bit for bit
    tmp = torch.empty(n, c, h, w, dtype=torch.float32, device="cuda")
    _ok(engine, "ss4k_glue_finalize", *args, None, _p(tmp), 0)
    two = torch.full_like(fused, 9)
    _ok(engine, "ss4k_glue_bicubic_u8", _p(tmp), n, c, h, w, _p(two), oh, ow, round_u8)
    assert torch.equal(fused, two)


def test_finalize_bicubic_u8_rejects_factors_beyond_its_patch(engine):
    hr = torch.zeros(1, 3, 272, 240, dtype=torch.float16, device="cuda")
    out = torch.zeros(100 * 120 * 3, dtype=torch.uint8, device="cuda")
    base = (_p(hr), 1, 1, 3)
    assert _call(engine, "ss4k_glue_finalize_bicubic_u8", *base, 272, 240, None, 0, 0, None, None, 1.0, 1.0, _p(out),
                 100, 120, 0) == E_INVALID                                               # fy = 2.72
    assert _call(engine, "ss4k_glue_finalize_bicubic_u8", *base, 200, 217, None, 0, 0, None, None, 1.0, 1.0, _p(out),
                 100, 100, 0) == E_INVALID                                               # fx = 2.17
    assert _call(engine, "ss4k_glue_finalize_bicubic_u8", *base, 200, 216, None, 0, 0, None, None, 1.0, 1.0, _p(out),
                 100, 100, 0) == L.OK                                                    # fx = 2.16


# ---------------------------------------------------------------- sharpen_blend
@pytest.mark.parametrize("fmt,n,c,h,w,strength,opacity,other_fmt", [
    (1, 1, 3, 48, 64, 0.00002, 0.8, 0),    # the denoise blend of upscale_single
    (0, 1, 3, 37, 53, 0.00007, 1.0, None),  # the HR sharpen of upscale_single
    (2, 2, 3, 2, 2, 1.0, 0.8, 1),           # smallest image the 3x3 reflect takes; strength 1 drives the clamp
    (1, 2, 3, 19, 33, 0.0, 0.8, 2),
    (0, 2, 3, 18, 30, 1.0, 0.8, 3),         # NV12 other
    (2, 1, 3, 31, 2, 0.00002, 0.8, None),
    (1, 1, 1, 2, 9, 1.0, 1.0, None),
])
def test_sharpen_blend(engine, fmt, n, c, h, w, strength, opacity, other_fmt):
    x_dev, x64 = _as_fmt(_noise(n, c, h, w, 13), fmt)
    o_dev, o64 = _other(other_fmt, n, c, h, w, 14)
    out = torch.full((n, c, h, w), float("nan"), dtype=torch.float32, device="cuda")
    _ok(engine, "ss4k_glue_sharpen_blend", _p(x_dev), fmt, n, c, h, w, strength, opacity, _p(o_dev),
        other_fmt if other_fmt is not None else 0, _p(out))
    ref, mag = _sharpen64(x64, strength, opacity, o64)
    _assert_f32(out, ref, mag, 1e-6, "sharpen_blend")


# ---------------------------------------------------------------- sharpen_blend_act
def _act64(x64, strength, opacity, o64, us, pitch):
    """The sharpen / blend value in the activation layout: pixel_unshuffle(us) channel order, NHWC, zero padding."""
    v, _ = _sharpen64(x64, strength, opacity, o64)
    v = F.pixel_unshuffle(v, us).permute(0, 2, 3, 1)
    return torch.cat([v, torch.zeros(*v.shape[:3], pitch - v.shape[-1], dtype=v.dtype)], dim=-1)


def _act_call(engine, x_dev, fmt, n, c, h, w, strength, opacity, o_dev, other_fmt, us, pitch, bf16):
    out = torch.full((n, h // us, w // us, pitch), -1, dtype=torch.int16, device="cuda")   # all bits set
    _ok(engine, "ss4k_glue_sharpen_blend_act", _p(x_dev), fmt, n, c, h, w, strength, opacity, _p(o_dev),
        other_fmt if other_fmt is not None else 0, _p(out), us, pitch, bf16)
    return out


def _check_act(out, ref, creal, bf16, what):
    vals = out.view(torch.bfloat16 if bf16 else torch.float16)
    _assert_16(vals[..., :creal], ref[..., :creal], bf16, what)
    assert (out[..., creal:] == 0).all(), "padding channels must be exactly zero"


@pytest.mark.parametrize("fmt,n,c,h,w,us,pitch,bf16,other_fmt", [
    (1, 2, 3, 10, 14, 1, 8, 0, None),     # pitch = 3 rounded up to 8
    (0, 1, 3, 12, 18, 2, 16, 1, 0),       # bf16, x float: generic kernel
    (2, 1, 3, 16, 24, 4, 48, 0, 3),       # unshuffle 4, x uint8, NV12 other
    (1, 2, 3, 8, 12, 4, 64, 1, 2),
    (1, 1, 1, 6, 10, 2, 64, 0, 1),        # C = 1
    (0, 3, 3, 2, 2, 1, 64, 0, 2),
    (1, 2, 3, 10, 14, 2, 16, 0, 1),       # half other: generic kernel at the hand-over's geometry
])
def test_sharpen_blend_act_generic(engine, fmt, n, c, h, w, us, pitch, bf16, other_fmt):
    x_dev, x64 = _as_fmt(_noise(n, c, h, w, 15), fmt)
    o_dev, o64 = _other(other_fmt, n, c, h, w, 16)
    out = _act_call(engine, x_dev, fmt, n, c, h, w, 0.00002, 0.8, o_dev, other_fmt, us, pitch, bf16)
    _check_act(out, _act64(x64, 0.00002, 0.8, o64, us, pitch), c * us * us, bf16, "sharpen_blend_act")


@pytest.mark.parametrize("n,h,w", [(3, 2, 2), (2, 18, 34)])
@pytest.mark.parametrize("pitch", [16, 24, 64])
@pytest.mark.parametrize("other_fmt", [None, 2, 3])
def test_sharpen_blend_act_us2(engine, monkeypatch, n, h, w, pitch, other_fmt):
    """The x2 hand-over kernel (half NCHW in, pixel_unshuffle(2), fp16 out) against the fp64 value and, bit for bit,
    against the generic kernel (SS4K_GLUE_GENERIC, read on every call)."""
    x_dev, x64 = _as_fmt(_noise(n, 3, h, w, 17, -0.05, 1.05), 1)
    o_dev, o64 = _other(other_fmt, n, 3, h, w, 18)
    args = (engine, x_dev, 1, n, 3, h, w, 0.00002, 0.8, o_dev, other_fmt, 2, pitch, 0)
    monkeypatch.delenv("SS4K_GLUE_GENERIC", raising=False)
    fast = _act_call(*args)
    _check_act(fast, _act64(x64, 0.00002, 0.8, o64, 2, pitch), 12, False, "sharpen_blend_act us2")
    monkeypatch.setenv("SS4K_GLUE_GENERIC", "1")
    assert torch.equal(fast, _act_call(*args))


# ---------------------------------------------------------------- geometry the reference refuses
def _inside(n_elems, dtype):
    """A device buffer as a view 4096 elements into a larger zeroed allocation: a build without the geometry checks
    then reads only memory this test owns."""
    return _at_offset(torch.zeros(n_elems, dtype=dtype, device="cuda"), 4096, pad=4096)


def test_glue_entries_reject_geometry_the_reference_refuses(engine):
    f32, f16, u8 = torch.float32, torch.float16, torch.uint8
    img, img16, img8 = _inside(4096, f32), _inside(4096, f16), _inside(4096, u8)
    out, out16, out8 = _inside(4096, f32), _inside(4096, f16), _inside(4096, u8)
    kern, sums = _inside(17 * 17, f32), _inside(64, torch.float64)
    rej = []

    def blur(ksize, n, c, h, w):
        return _call(engine, "ss4k_glue_blur_diff", _p(img), _p(img), _p(out), _p(kern), ksize, n, c, h, w, None, None, 0.0, 0.0)

    # reflect padding of radius ksize // 2 needs ksize // 2 < h and < w (F.pad(mode='reflect') raises otherwise)
    rej += [("blur 17 on 8 wide", blur(17, 1, 3, 9, 8)), ("blur 17 on 8 tall", blur(17, 1, 3, 8, 9)),
            ("blur 3 on 1 tall", blur(3, 1, 1, 1, 5)), ("blur even ksize", blur(4, 1, 3, 9, 9)),
            ("blur ksize 0", blur(0, 1, 3, 9, 9)), ("blur n 0", blur(3, 0, 3, 9, 9)), ("blur c 0", blur(3, 1, 0, 9, 9))]
    assert blur(17, 1, 3, 9, 9) == L.OK

    def sharpen(h, w):
        return _call(engine, "ss4k_glue_sharpen_blend", _p(img16), 1, 1, 3, h, w, 0.00002, 0.8, _p(img), 0, _p(out))

    def act(h, w, us):
        return _call(engine, "ss4k_glue_sharpen_blend_act", _p(img16), 1, 1, 3, h, w, 0.00002, 0.8, _p(img8), 2, _p(out16),
                     us, 64, 0)

    rej += [("sharpen 1 tall", sharpen(1, 8)), ("sharpen 1 wide", sharpen(8, 1)),
            ("act 1 tall", act(1, 8, 1)), ("act 1 wide", act(8, 1, 1))]
    assert sharpen(2, 2) == L.OK and act(2, 2, 2) == L.OK

    def finalize(dh, dw):
        return _call(engine, "ss4k_glue_finalize", _p(img16), 1, 1, 3, 8, 8, _p(img), dh, dw, None, None, 0.0, 0.0, _p(out8),
                     None, 0)

    def finalize_bicubic(dh, dw):
        return _call(engine, "ss4k_glue_finalize_bicubic_u8", _p(img16), 1, 1, 3, 8, 8, _p(img), dh, dw, None, None, 0.0, 0.0,
                     _p(out8), 9, 9, 0)

    rej += [("finalize dh 0", finalize(0, 2)), ("finalize dw 0", finalize(2, 0)),
            ("finalize_bicubic dh 0", finalize_bicubic(0, 2)), ("finalize_bicubic dw 0", finalize_bicubic(2, 0))]
    assert finalize(1, 1) == L.OK and finalize_bicubic(1, 1) == L.OK

    def pool(n, c, h, w, oh, ow):
        return _call(engine, "ss4k_glue_area_pool", _p(img), 0, n, c, h, w, _p(out), oh, ow)

    def bicubic(n, c, h, w, oh, ow):
        return _call(engine, "ss4k_glue_bicubic_u8", _p(img), n, c, h, w, _p(out8), oh, ow, 0)

    for i, dims in enumerate([(0, 3, 8, 8, 4, 4), (1, 0, 8, 8, 4, 4), (1, 3, 0, 8, 4, 4), (1, 3, 8, 0, 4, 4),
                              (1, 3, 8, 8, 0, 4), (1, 3, 8, 8, 4, -1)]):
        rej += [(f"area_pool {dims}", pool(*dims)), (f"bicubic_u8 {dims}", bicubic(*dims))]
    assert pool(1, 3, 8, 8, 4, 4) == L.OK and bicubic(1, 3, 8, 8, 4, 4) == L.OK
    wrong = [what for what, rc in rej if rc != E_INVALID]
    assert not wrong, wrong


def test_service_refuses_colour_match_narrower_than_its_blur(engine):
    """The still-image server (lr_hr_resize=False) with SRVGG x4 on an 18 x 17 image: the net's output is 72 x 68, so the
    colour match pools to 9 x 8 and blurs with radius 8.  The reference's F.pad(mode='reflect') raises there; the engine
    must raise as well (Ss4kError is a RuntimeError), not read outside the pooled image, and serve the next image."""
    torch.manual_seed(0)
    net = srvgg.SRVGGNetCompact(3, 3, 64, 16, 4).eval()
    narrow, square = _frames_u8(1, 18, 17, 21), _frames_u8(1, 18, 18, 22)
    with pytest.raises(RuntimeError):
        glue.upscale_multi(narrow, net, lr_shape=(720, 1280), output_shape=None, lr_hr_resize=False)
    svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, model_name='realesr-animevideov3',
                                        state_dict=net.state_dict(), batch_size=1, lr_hr_resize=False)
    svc.proc_init()
    with pytest.raises(RuntimeError):
        svc.upscale(narrow.cuda())
    torch.cuda.synchronize()
    got = svc.upscale(square.cuda()).cpu()
    want_u8, want_q = glue.upscale_multi(square, net, lr_shape=(720, 1280), output_shape=None, lr_hr_resize=False,
                                         return_float=True)
    assert got.shape == want_u8.shape == (1, 72, 72, 3)
    # the net runs in fp16 here: the service tests' gate on the float frame (|engine - oracle| <= 2/255)
    e = got.float() - want_q
    assert e.max().item() <= 2.0 and e.min().item() > -3.0


def _frames_u8(n, h, w, seed):
    return (_smooth(n, 3, h, w, seed) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()


# ---------------------------------------------------------------- the reference's golden glue outputs
def _golden_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


def _near_golden(got, want, want_q, what):
    """got / want: uint8 frames; want_q: the oracle's float frame (x255) in front of the truncating cast.  At most one
    level apart, only where the float frame is within EPS_U8 of an integer, on at most 1e-3 of the values."""
    got, want = torch.as_tensor(got).int(), torch.as_tensor(want).int()
    d = (got.cpu() - want).abs()
    frac = want_q.double() - torch.floor(want_q.double())
    dist = torch.minimum(frac, 1.0 - frac)
    far = dist[d > 0].max().item() if (d > 0).any() else 0.0
    print(f"{what}: {int((d > 0).sum())} of {d.numel()} values one level off, largest boundary distance {far:.2e}")
    assert d.max().item() <= 1 and far <= EPS_U8 and (d > 0).float().mean().item() <= 1e-3, (what, far)


@pytest.fixture(scope="module")
def golden_service(engine):
    """FsrcnnUpscalerService with its nets replaced by the stand-ins the golden glue outputs were made with."""
    torch.manual_seed(0)
    net = srvgg.SRVGGNetCompact(3, 3, 64, 16, 4).eval()
    svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, model_name='realesr-animevideov3',
                                        state_dict=net.state_dict(), batch_size=2)
    svc.proc_init()
    mg = _golden_module()
    model, den = mg.glue_models()
    svc.model = model                               # float32 out, as in the golden run
    # uint8 NHWC frames are read as the reference's permute / 255; the glue wants a contiguous NCHW tensor
    svc._run_model = lambda lr: model(lr.permute(0, 3, 1, 2) / 255.0 if lr.dtype == torch.uint8 else lr).contiguous()
    return svc, mg, model, den


def test_service_glue_matches_reference_golden(golden_service):
    svc, mg, model, den = golden_service
    g = np.load(os.path.join(GOLD, "glue.npz"))
    frames = torch.from_numpy(g["frames"])
    svc.single_mode, svc.denoising, svc.denoise_model = False, False, None
    for i, (lr_shape, out_shape) in enumerate(mg.GLUE_MULTI_CASES):
        svc.lr_shape, svc.output_shape = tuple(lr_shape), out_shape
        got = svc.upscale(frames.cuda())
        _, q = glue.upscale_multi(frames.clone(), model, lr_shape=lr_shape, output_shape=out_shape, return_float=True)
        _near_golden(got, g[f"multi{i}"], q, f"multi{i}")
    svc.single_mode, svc.denoise_rate = True, 0.75
    svc.lr_shape, svc.output_shape = tuple(mg.GLUE_SINGLE_LR), mg.GLUE_SINGLE_OUT
    for i, use_den in enumerate((False, True)):
        svc.denoising, svc.denoise_model, svc.lr_prev = use_den, den if use_den else None, None
        for fi in range(2):   # first frame, then the steady-state noise map
            got = svc.upscale(frames[fi:fi + 1].cuda())[0]
            _, q = glue.upscale_single(frames[fi].clone(), model, lr_shape=mg.GLUE_SINGLE_LR, output_shape=mg.GLUE_SINGLE_OUT,
                                       denoise_model=den if use_den else None, denoise_rate=0.75, first_frame=fi == 0,
                                       return_float=True)
            _near_golden(got, g[f"single{i}_{fi}"], q, f"single{i}_{fi}")
