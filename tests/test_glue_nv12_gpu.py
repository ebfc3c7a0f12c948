"""NV12 output of the colour-match finalising kernels (csrc/glue.cu): ss4k_glue_finalize_bicubic_nv12 and
ss4k_glue_finalize_nv12 must write exactly the bytes of the uint8 RGB entry with the same arguments followed by
ss4k_rgb_to_nv12, and nothing past the frames.  Each NV12 result sits at the front of a larger allocation whose tail
(the canary) must stay untouched."""
import pytest
import torch

from ss4k_b200 import _lib as L
from tests.test_glue_gpu import E_INVALID, _call, _diff, _diff_shape, _match_inputs, _ok, _p, _staged_tiles, _stats_dev

pytestmark = pytest.mark.gpu

CANARY = 0xA5


def _nv12_out(n, oh, ow, offset=0, pad=4096):
    """(whole allocation, NV12 view [n, oh*3/2, ow] `offset` bytes into it); the rest of the allocation holds CANARY."""
    size = n * oh * ow * 3 // 2
    buf = torch.full((offset + size + pad,), CANARY, dtype=torch.uint8, device="cuda")
    return buf, buf[offset:offset + size].view(n, oh * 3 // 2, ow)


def _canary_intact(buf, n, oh, ow):
    size = n * oh * ow * 3 // 2
    return bool((buf[size:] == CANARY).all())


def _via_rgb(engine, rgb):
    n, oh, ow, _ = rgb.shape
    return engine.rgb_to_nv12(rgb).view(n, oh * 3 // 2, ow)


def _inputs(engine, fmt, n, h, w, dmode, seed, sums=True):
    """(the entries' leading arguments, the device tensors they point to).  The caller keeps the tensors alive for as
    long as it uses the pointers: freed, their memory goes back to the caching allocator and the next output buffer may
    be placed on top of it."""
    hr_dev, hr64, lr_dev, lr64 = _match_inputs(n, 3, h, w, 6, 8, seed)
    if fmt == 0:
        hr_dev = hr_dev.float()
    hs = ls = None
    if sums:
        hs, ls = _stats_dev(engine, hr_dev, fmt, n, 3, h, w), _stats_dev(engine, lr_dev, 0, n, 3, 6, 8)
    dshape = _diff_shape(dmode, h, w)
    d_dev, _ = _diff(n, 3, dshape, seed + 1)
    dh, dw = dshape if dshape else (0, 0)
    args = (_p(hr_dev), fmt, n, 3, h, w, _p(d_dev), dh, dw, _p(hs), _p(ls), float(h * w), 48.0)
    return args, (hr_dev, lr_dev, hs, ls, d_dev)


# ---------------------------------------------------------------- finalize_bicubic_nv12
@pytest.mark.parametrize("fmt,n,h,w,oh,ow,dmode,round_u8", [
    (1, 2, 96, 128, 100, 140, "1/8", 0),    # staged diff rows; OW % 32 = 12, OH % 8 = 4 (4-row last tile)
    (1, 1, 160, 240, 80, 120, "1/8", 1),    # downscale exactly 2, staged
    (1, 2, 360, 640, 180, 320, "1/8", 0),   # the live default's 2x downscale in miniature
    (0, 2, 96, 128, 48, 64, "1/2", 0),      # diff at H/2: un-staged tiles
    (1, 1, 64, 96, 100, 152, "full", 1),    # diff at H, upscaling: un-staged
    (1, 1, 270, 200, 100, 100, "1/8", 0),   # fy = 2.7: just inside the patch guard
    (0, 1, 50, 70, 38, 44, None, 0),        # no diff; OH % 8 = 6 (6-row last tile)
    (1, 2, 72, 136, 146, 272, None, 1),     # upscaling; OH % 8 = 2 (2-row last tile)
])
def test_finalize_bicubic_nv12(engine, fmt, n, h, w, oh, ow, dmode, round_u8):
    args, keep = _inputs(engine, fmt, n, h, w, dmode, 31)   # noqa: F841 (keeps the inputs alive)
    if dmode is not None:
        some_staged, some_not = _staged_tiles(h, oh, args[7])
        assert (some_staged and not some_not) if dmode == "1/8" else some_not
    rgb = torch.full((n, oh, ow, 3), 7, dtype=torch.uint8, device="cuda")
    _ok(engine, "ss4k_glue_finalize_bicubic_u8", *args, _p(rgb), oh, ow, round_u8)
    buf, nv = _nv12_out(n, oh, ow)
    _ok(engine, "ss4k_glue_finalize_bicubic_nv12", *args, _p(nv), oh, ow, round_u8)
    assert torch.equal(nv, _via_rgb(engine, rgb))
    assert _canary_intact(buf, n, oh, ow)


# ---------------------------------------------------------------- finalize_nv12
@pytest.mark.parametrize("fmt,n,h,w,dmode,round_u8,sums", [
    (1, 2, 64, 96, "1/8", 0, True),       # the service's shape of the call
    (1, 2, 192, 320, "1/8", 0, True),     # RRDBNet x2 on a 96 x 160 frame
    (0, 3, 16, 20, "full", 1, True),      # full-size diff; n = 3; W % 32 != 0
    (1, 2, 72, 100, None, 0, False),      # no diff, NULL sums; W % 32 = 4
    (1, 3, 26, 44, "1/8", 0, True),       # n = 3; H % 8 = 2, W % 32 = 12
    (0, 1, 38, 36, "1/2", 1, True),
])
def test_finalize_nv12(engine, fmt, n, h, w, dmode, round_u8, sums):
    args, keep = _inputs(engine, fmt, n, h, w, dmode, 41, sums)   # noqa: F841 (keeps the inputs alive)
    rgb = torch.full((n, h, w, 3), 7, dtype=torch.uint8, device="cuda")
    _ok(engine, "ss4k_glue_finalize", *args, _p(rgb), None, round_u8)
    buf, nv = _nv12_out(n, h, w)
    _ok(engine, "ss4k_glue_finalize_nv12", *args, _p(nv), round_u8)
    assert torch.equal(nv, _via_rgb(engine, rgb))
    assert _canary_intact(buf, n, h, w)


# ---------------------------------------------------------------- rejected geometry
def test_nv12_entries_reject_what_nv12_cannot_hold(engine):
    hr = torch.zeros(1, 3, 272, 240, dtype=torch.float16, device="cuda")
    buf = torch.full((1 << 20,), CANARY, dtype=torch.uint8, device="cuda")
    out, odd = buf[4096:], buf[4097:]

    def fb(c, h, w, oh, ow, o=out):
        return _call(engine, "ss4k_glue_finalize_bicubic_nv12", _p(hr), 1, 1, c, h, w, None, 0, 0, None, None, 1.0, 1.0, _p(o),
                     oh, ow, 0)

    def fin(c, h, w, o=out):
        return _call(engine, "ss4k_glue_finalize_nv12", _p(hr), 1, 1, c, h, w, None, 0, 0, None, None, 1.0, 1.0, _p(o), 0)

    rej = [("fb odd oh", fb(3, 200, 200, 99, 100)), ("fb ow % 4", fb(3, 200, 200, 100, 98)), ("fb c 2", fb(2, 200, 200, 100, 100)),
           ("fb c 4", fb(4, 200, 200, 100, 100)), ("fb misaligned", fb(3, 200, 200, 100, 100, odd)),
           ("fb fy 2.72", fb(3, 272, 240, 100, 120)), ("fb fx 2.17", fb(3, 200, 217, 100, 100)),
           ("fin odd h", fin(3, 199, 200)), ("fin w % 4", fin(3, 200, 198)), ("fin c 1", fin(1, 200, 200)),
           ("fin misaligned", fin(3, 200, 200, odd)),
           ("fin dh 0", _call(engine, "ss4k_glue_finalize_nv12", _p(hr), 1, 1, 3, 8, 8, _p(hr), 0, 2, None, None, 1.0, 1.0,
                              _p(out), 0))]
    wrong = [what for what, rc in rej if rc != E_INVALID]
    assert not wrong, wrong
    assert bool((buf == CANARY).all())                                  # nothing was written
    assert fb(3, 200, 216, 100, 100) == L.OK and fin(3, 200, 200) == L.OK   # fx = 2.16 and a plain call pass
