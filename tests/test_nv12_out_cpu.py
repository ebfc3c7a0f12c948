"""NV12 output of RRDBNet plans, host side: the planner's lowering (ss4k_plan_dry), the formats it refuses, the
pair-aligned row split of the streaming kernel's NV12 store (restated from csrc/conv_stream.cu) and the Python layer's
output shape / dtype."""
import ctypes

import pytest
import torch

import ss4k_b200
from ss4k_b200 import _lib as L
from ss4k_b200 import engine as E

K_OUT_NV12 = 8          # csrc/conv_params.h OutMode
K_OUT_U8NHWC = 6
E_INVALID = -1
TILE_W = 128            # pixels per strip (kTileW)


def _dry_rc(cfg):
    lib = L.load()
    out = ctypes.c_void_p()
    rc = lib.ss4k_plan_dry(ctypes.byref(cfg), ctypes.byref(out))
    if rc == 0:
        lib.ss4k_free(out)
    return rc


@pytest.mark.parametrize("scale,h,w", [(2, 96, 128), (4, 96, 128), (2, 70, 46), (4, 70, 46), (2, 720, 1280)])
def test_rrdb_nv12_plan_marks_conv_last(lib, scale, h, w):
    prog = ss4k_b200.plan_dry(ss4k_b200.make_cfg(0, L.ARCH_RRDB, 3, h, w, scale=scale, depth=2, out_fmt=L.FMT_NV12))
    assert prog["out_fmt"] == L.FMT_NV12
    assert (prog["out_h"], prog["out_w"]) == (h * scale, w * scale)
    last = prog["steps"][-1]
    assert last["kind"] == "conv" and last["name"] == "conv_last"
    assert last["out_mode"] == K_OUT_NV12 and last["cout"] == 3 and last["out_buf"] == -3
    # every other conv is lowered exactly as for uint8 RGB output
    ref = ss4k_b200.plan_dry(ss4k_b200.make_cfg(0, L.ARCH_RRDB, 3, h, w, scale=scale, depth=2, out_fmt=L.FMT_U8_NHWC))
    assert ref["steps"][-1]["out_mode"] == K_OUT_U8NHWC
    assert len(ref["steps"]) == len(prog["steps"])
    for a, b in zip(ref["steps"][:-1], prog["steps"][:-1]):
        assert a == b
    assert {k: v for k, v in ref["steps"][-1].items() if k != "out_mode"} == \
        {k: v for k, v in last.items() if k != "out_mode"}


@pytest.mark.parametrize("arch,scale", [(L.ARCH_SRVGG, 4), (L.ARCH_SRVGG, 2), (L.ARCH_BSVD, 1)])
def test_nv12_out_rejected_for_srvgg_and_bsvd(lib, arch, scale):
    cfg = ss4k_b200.make_cfg(0, arch, 2, 64, 128, scale=scale, out_fmt=L.FMT_NV12)
    assert _dry_rc(cfg) == E_INVALID
    with pytest.raises(L.Ss4kError, match="NV12 output is for RRDBNet plans"):
        ss4k_b200.plan_dry(cfg)


# ---- pair-aligned row split of the NV12 store (conv3x3_stream_kernel: u0 / u1 with pair_sh = 1)
def _split(total, grid, pair):
    sh = 1 if pair else 0
    return [((b * (total >> sh)) // grid << sh, ((b + 1) * (total >> sh)) // grid << sh) for b in range(grid)]


def _bands(u0, u1, H):
    """Start rows of the bands (runs of rows inside one strip) a CTA with units [u0, u1) walks, and the row counter q at
    each (conv_stream.cu next_band)."""
    out, u, q = [], u0, 0
    while u < u1:
        y = u % H
        ye = min(H, y + (u1 - u))
        out.append((y, q))
        q += ye - y
        u += ye - y
    return out


# output geometries of the GPU tests: (batch, out_h, out_w)
GEOMS = [(n, h * s, w * s) for n in (1, 3) for s in (2, 4) for (h, w) in ((96, 128), (70, 46))] + \
        [(n, 1440, 2560) for n in (1, 3)] + [(1, 2160, 3840), (2, 1080, 1920)]


@pytest.mark.parametrize("n,H,W", GEOMS)
def test_pair_split_starts_every_band_on_an_even_row(n, H, W):
    strips = (W + TILE_W - 1) // TILE_W
    total = n * strips * H     # chunks == 1 for conv_last (cout 3 -> NOUT 16)
    assert H % 2 == 0 and W % 4 == 0
    for grid in range(1, 149):
        runs = _split(total, grid, pair=True)
        assert runs[0][0] == 0 and runs[-1][1] == total
        for (a0, a1), (b0, _) in zip(runs, runs[1:]):
            assert a1 == b0 and a0 <= a1
        for u0, u1 in runs:
            assert u0 % 2 == 0 and u1 % 2 == 0
            for y, q in _bands(u0, u1, H):
                # the row's parity is the row counter's parity: row 2j -> the parity-0 warp, 2j+1 -> the parity-1 warp
                assert y % 2 == 0 and q % 2 == 0


def test_old_split_would_start_some_cta_on_an_odd_row():
    """The geometries above include row totals for which the plain even split gives a CTA an odd first row (which the
    NV12 store must not see): proves the pair split is exercised, not a no-op."""
    hits = 0
    for n, H, W in GEOMS:
        total = n * ((W + TILE_W - 1) // TILE_W) * H
        grid = min(total, 148)
        if any(y % 2 for u0, u1 in _split(total, grid, pair=False) for y, _ in _bands(u0, u1, H)):
            hits += 1
    assert hits >= len(GEOMS) // 2


# ---- Python layer
def test_plan_out_shape_and_dtype_for_nv12():
    assert E._OUT_DTYPES[L.FMT_NV12] == torch.uint8
    plan = E.Plan.__new__(E.Plan)      # the shape logic only: no device needed
    plan.out_nchw = (3, 3, 1440, 2560)
    plan.cfg = ss4k_b200.make_cfg(0, L.ARCH_RRDB, 3, 720, 1280, scale=2, out_fmt=L.FMT_NV12)
    assert plan.out_shape() == (3, 2160, 2560)
    plan.cfg = ss4k_b200.make_cfg(0, L.ARCH_RRDB, 3, 720, 1280, scale=2, out_fmt=L.FMT_U8_NHWC)
    assert plan.out_shape() == (3, 1440, 2560, 3)
    plan.cfg = ss4k_b200.make_cfg(0, L.ARCH_RRDB, 3, 720, 1280, scale=2, out_fmt=L.FMT_F16_NCHW)
    assert plan.out_shape() == (3, 3, 1440, 2560)
    # NV12 frames are half the bytes of uint8 RGB
    n, c, h, w = plan.out_nchw
    assert 2 * torch.Size(E.out_shape_of(L.FMT_NV12, n, c, h, w)).numel() == torch.Size(E.out_shape_of(L.FMT_U8_NHWC, n, c, h, w)).numel()
