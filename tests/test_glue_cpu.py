"""Host-side bound behind ss4k_glue_finalize_bicubic_u8 (csrc/glue.cu): the entry accepts a resize when
h/oh * (kFbTh - 1) + 5 <= kFbMaxH and w/ow * (kFbTw - 1) + 5 <= kFbMaxW, and the kernel then finalises a source patch of
ph x pw pixels into a fixed kFbMaxH x kFbMaxW shared-memory array.  This emulates the kernel's float32 patch bounds
(py0 / py1 / px0 / px1) for every accepted size pair up to a few hundred pixels and proves the patch fits, and that every
bicubic tap of the tile lands inside it."""
import numpy as np
import pytest

TW, TH, MAX_W, MAX_H = 32, 8, 72, 24   # kFbTw, kFbTh, kFbMaxW, kFbMaxH
SIZES = np.arange(1, 321)


def _accepted(n_in, n_out, tile, max_patch):
    """The entry's guard, in double like the host code."""
    return (np.asarray(n_in, dtype=np.float64) / n_out) * (tile - 1) + 5.0 <= max_patch


def _src(o, f, fused):
    """float32 (o + 0.5f) * f - 0.5f, with or without the multiply-add contracted into one rounding (nvcc contracts by
    default; both forms are checked so the bound does not rest on that choice).  The float64 product of two float32
    values is exact, and so is the sum with -0.5 at these magnitudes: one cast is exactly one fmaf rounding."""
    a = o.astype(np.float32) + np.float32(0.5)
    if fused:
        return (a.astype(np.float64) * f.astype(np.float64) - 0.5).astype(np.float32)
    return (a * f).astype(np.float32) - np.float32(0.5)


def _patch_extent(n_in, n_out, tile, fused):
    """Largest patch extent over every tile and the extreme tap offsets relative to the patch origin, for all n_in
    (vector) at one n_out.  Returns (max extent per n_in, min tap offset, max tap offset - extent)."""
    f = (n_in.astype(np.float32) / np.float32(n_out)).astype(np.float32)[:, None]          # fy = (float)H / OH
    o0 = np.arange(0, n_out, tile)[None, :]
    o1 = np.minimum(o0 + tile, n_out) - 1
    p0 = np.floor(_src(o0, f, fused)).astype(np.int64) - 1
    p1 = np.floor(_src(o1, f, fused)).astype(np.int64) + 2
    ext = (p1 - p0 + 1).max(axis=1)
    # taps of every output pixel: floor(s) - 1 .. floor(s) + 2 relative to its tile's p0
    o = np.arange(n_out)[None, :]
    i = np.floor(_src(o, f, fused)).astype(np.int64)
    base = p0[:, o[0] // tile]
    lo = (i - 1 - base).min(axis=1)
    hi = (i + 2 - base - (p1 - p0 + 1)[:, o[0] // tile]).max(axis=1)
    return ext, lo, hi


@pytest.mark.parametrize("axis", ["y", "x"])
@pytest.mark.parametrize("fused", [True, False])
def test_finalize_bicubic_patch_fits_shared_memory(axis, fused):
    tile, max_patch = (TH, MAX_H) if axis == "y" else (TW, MAX_W)
    checked = 0
    worst = 0
    for n_out in SIZES:
        n_in = SIZES[_accepted(SIZES, n_out, tile, max_patch)]
        if n_in.size == 0:
            continue
        ext, lo, hi = _patch_extent(n_in, n_out, tile, fused)
        assert ext.max() <= max_patch, (axis, n_out, n_in[ext.argmax()], ext.max())
        assert lo.min() >= 0 and hi.max() < 0, (axis, n_out)   # every tap row / column is inside the staged patch
        worst = max(worst, int(ext.max()))
        checked += n_in.size
    print(f"{axis}: {checked} accepted size pairs, largest patch extent {worst} (limit {max_patch})")
    # the guard admits factors up to (max_patch - 5) / (tile - 1): 2.71 along y, 2.16 along x
    assert checked > 40000 and worst > max_patch - 4


def test_guard_limits():
    """Factors the GPU tests use on either side of the guard."""
    assert _accepted(np.array([270]), 100, TH, MAX_H)[0]          # fy = 2.7: inside
    assert not _accepted(np.array([272]), 100, TH, MAX_H)[0]      # fy = 2.72: outside
    assert _accepted(np.array([216]), 100, TW, MAX_W)[0]          # fx = 2.16: inside
    assert not _accepted(np.array([217]), 100, TW, MAX_W)[0]      # fx = 2.17: outside
