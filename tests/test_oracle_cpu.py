"""Pins the CPU oracle (oracle/) to the reference.

  * golden fixtures (tests/golden/*.npz) are outputs of the REFERENCE's own nn.Modules, minted by
    tests/golden/make_golden.py in the build container; the oracle must rebuild the same weights
    from the seed (checksums) and reproduce the outputs.
  * when /root/reference is present (build container only, never the GPU box) the restatements are
    additionally compared with the live reference modules on fresh seeds.
  * the service glue (oracle/glue.py) is pinned to the reference's own upscale_multi / upscale_single code, cut out of
    src/upscale/fsrcnn_upscaler.py by its AST (the module itself cannot be imported) and run on the CPU in fp32.
  * RRDBNet lives in un-vendored pip `basicsr`: pinned only by its known-answer parameter counts and
    state-dict key names (SURVEY.md Appendix A) -> parity unpinned, stated in DESIGN.md.
"""
import os

import numpy as np
import pytest
import torch

from oracle import bsvd, glue, rrdbnet, srvgg
from oracle import reference_import as ri

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_ref = pytest.mark.skipif(not ri.available(), reason="/root/reference not present (GPU box)")


def _check_weights(sd, g):
    keys = list(g["keys"])
    assert sorted(sd.keys()) == keys
    sums = g["sums"]
    for i, k in enumerate(keys):
        t = sd[k].double()
        assert abs(t.sum().item() - sums[i, 0]) <= 1e-9 * max(1.0, abs(sums[i, 0])), k
        assert abs((t ** 2).sum().item() - sums[i, 1]) <= 1e-9 * max(1.0, abs(sums[i, 1])), k


@pytest.mark.parametrize("nconv", [16, 32])
def test_srvgg_golden(nconv):
    g = np.load(os.path.join(GOLD, f"srvgg{nconv}_x4.npz"))
    torch.set_num_threads(1)
    torch.manual_seed(int(g["seed"]))
    net = srvgg.SRVGGNetCompact(3, 3, 64, nconv, 4).eval()
    _check_weights(net.state_dict(), g)
    with torch.no_grad():
        y = net(torch.from_numpy(g["x"]))
    assert tuple(y.shape) == (1, 3, 48, 80)
    assert (y - torch.from_numpy(g["y"])).abs().max().item() <= 1e-6


@pytest.mark.parametrize("frames", [5, 1])
def test_bsvd_golden(frames):
    g = np.load(os.path.join(GOLD, f"bsvd32_f{frames}.npz"))
    torch.set_num_threads(1)
    sd = bsvd.build_bsvd32(int(g["seed"]))
    _check_weights(sd, g)
    y = bsvd.bsvd_forward(sd, torch.from_numpy(g["x"]))
    want = torch.from_numpy(g["y"])
    assert y.shape == want.shape
    # outputs span +-14 with the constructor's kaiming init (SURVEY.md fact 10); conv accumulation
    # order may differ by a few ulp between the streaming reference and the clip formulation
    assert (y - want).abs().max().item() <= 2e-5 * max(1.0, want.abs().max().item())


def test_bsvd_f1_is_not_the_clip_function():
    """SURVEY.md fact 8: F=1 (what the service feeds) differs from the same frame inside a clip."""
    sd = bsvd.build_bsvd32(0)
    x = torch.rand(1, 4, 4, 16, 24, generator=torch.Generator().manual_seed(3))
    full = bsvd.bsvd_forward(sd, x)
    single = bsvd.bsvd_forward(sd, x[:, 1:2])
    assert (full[:, 1] - single[:, 0]).abs().max().item() > 1e-2


def test_bsvd_chunk_with_16_frame_halo_is_exact():
    """SURVEY.md fact 9 / section 8e: chunk + 16-frame halo reproduces the full clip (multi-GPU sharding)."""
    sd = bsvd.build_bsvd32(0)
    x = torch.rand(40, 4, 8, 8, generator=torch.Generator().manual_seed(5))
    full = bsvd.bsvd_clip(sd, x)
    lo, hi = 18, 22
    part = bsvd.bsvd_clip(sd, x[lo - 16:hi + 16])[16:16 + hi - lo]
    assert (part - full[lo:hi]).abs().max().item() <= 1e-5
    short = bsvd.bsvd_clip(sd, x[lo - 8:hi + 8])[8:8 + hi - lo]
    assert (short - full[lo:hi]).abs().max().item() > 1e-4


def test_rrdbnet_known_answers():
    """Parameter counts of the published architecture (SURVEY.md Appendix A) and key names."""
    def count(m):
        return sum(p.numel() for p in m.parameters())
    assert count(rrdbnet.RRDBNet(3, 3, 4, 64, 23, 32)) == 16_697_987
    assert count(rrdbnet.RRDBNet(3, 3, 2, 64, 23, 32)) == 16_703_171
    assert count(rrdbnet.RRDBNet(3, 3, 4, 64, 6, 32)) == 4_467_779
    net = rrdbnet.RRDBNet(3, 3, 2, 64, 2, 32)
    keys = set(net.state_dict().keys())
    for k in ("conv_first.weight", "body.0.rdb1.conv1.weight", "body.1.rdb3.conv5.bias", "conv_body.weight",
              "conv_up1.weight", "conv_up2.weight", "conv_hr.weight", "conv_last.bias"):
        assert k in keys
    x = torch.rand(1, 3, 10, 12)
    with torch.no_grad():
        assert tuple(net(x).shape) == (1, 3, 20, 24)
    # pixel_unshuffle channel order == torch's
    assert torch.equal(rrdbnet.pixel_unshuffle(x, 2), torch.nn.functional.pixel_unshuffle(x, 2))
    # upstream init: RDB convs are kaiming*0.1 with zero bias
    assert net.body[0].rdb1.conv1.bias.abs().max().item() == 0.0
    assert net.body[0].rdb1.conv1.weight.std().item() < 0.02


def test_tile_process_semantics():
    """RealESRGANer.tile_process: a pointwise 'model' must reproduce the untiled result exactly,
    and every output pixel is written once (no blending)."""
    x = torch.rand(1, 3, 37, 53)
    up = lambda t: torch.nn.functional.interpolate(t, scale_factor=2, mode="nearest")  # noqa: E731
    assert torch.equal(rrdbnet.tile_process(up, x, 2, 16, 5), up(x))


def test_glue_kernels_match_reference_formulas():
    """blur_ker / sharpen_ker weights (fsrcnn_upscaler.py:20-84)."""
    k = glue.sharpen_weight(0.00002)
    assert abs(k.sum().item() - 1.0) < 1e-6 and abs(k[0, 0, 1, 1].item() - (1 + 8 * 0.00002)) < 1e-6
    b = glue.blur_weight(17, 8.0)
    assert abs(b.sum().item() - 1.0) < 1e-5 and b[0, 0, 8, 8] == b.max()
    # the service's colour-match blur weights (service.py: gaussian_kernel(17, 8.0)) are blur_ker's
    from ss4k_b200 import service
    assert (service.gaussian_kernel(17, 8.0).double() - b[0, 0].double()).abs().max().item() <= 1e-9
    frames = torch.randint(0, 256, (2, 24, 32, 3), dtype=torch.uint8)
    up = lambda t: torch.nn.functional.interpolate(t, scale_factor=2, mode="bicubic")  # noqa: E731
    out = glue.upscale_multi(frames, up, lr_shape=(24, 32), output_shape=(48, 64))
    assert out.dtype == torch.uint8 and tuple(out.shape) == (2, 48, 64, 3)


def _glue_cases():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


def _same_u8(got, want):
    """uint8 outputs of two fp32 evaluations of the same graph: equal, up to a truncation flip of one level on a
    vanishing fraction of the values when the accumulation order of a library kernel differs between builds."""
    d = (torch.as_tensor(got).int() - torch.as_tensor(want).int()).abs()
    assert d.max().item() <= 1 and (d > 0).float().mean().item() <= 1e-3, (d.max().item(), (d > 0).float().mean().item())


def test_glue_golden():
    """oracle/glue.py against the uint8 outputs of the reference's OWN upscale_multi / upscale_single code
    (fsrcnn_upscaler.py:168-326, compiled from its source text by tests/golden/make_golden.py): area downscale branch,
    mean / std match, local colour match, bicubic resize, truncating uint8; single-frame path with and without the
    denoise branch, first and second frame."""
    mg = _glue_cases()
    g = np.load(os.path.join(GOLD, "glue.npz"))
    frames = torch.from_numpy(g["frames"])
    assert torch.equal(frames, mg.glue_frames())
    model, den = mg.glue_models()
    for i, (lr_shape, out_shape) in enumerate(mg.GLUE_MULTI_CASES):
        _same_u8(glue.upscale_multi(frames.clone(), model, lr_shape=lr_shape, output_shape=out_shape), g[f"multi{i}"])
    for i, use_den in enumerate((False, True)):
        for fi in range(2):
            got = glue.upscale_single(frames[fi].clone(), model, lr_shape=mg.GLUE_SINGLE_LR, output_shape=mg.GLUE_SINGLE_OUT,
                                      denoise_model=den if use_den else None, denoise_rate=0.75, first_frame=fi == 0)
            _same_u8(got, g[f"single{i}_{fi}"])


# ---------------------------------------------------------------- live reference (build container)
@needs_ref
def test_glue_matches_live_reference():
    """The same comparison against the reference's code executed live, on other shapes and seeds."""
    import warnings
    import torch.nn.functional as F
    warnings.simplefilter("ignore")
    ns = ri.load_fsrcnn_service_code()
    model = lambda t: F.interpolate(t.float(), scale_factor=4, mode="bilinear", align_corners=False) * 0.8 + 0.1  # noqa: E731
    den = lambda x: x[:, :, :3] * 0.9 + 0.05  # noqa: E731
    frames = torch.randint(0, 256, (3, 40, 72, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(11))
    for lr_shape, out_shape, resize in (((720, 1280), None, True), ((20, 36), (75, 133), True), ((20, 36), (75, 133), False)):
        svc = ri.make_reference_service(ns, model, lr_shape, out_shape, lr_hr_resize=resize)
        _same_u8(glue.upscale_multi(frames.clone(), model, lr_shape=lr_shape, output_shape=out_shape, lr_hr_resize=resize),
                 svc.upscale_multi(frames.clone()))
    svc = ri.make_reference_service(ns, model, (20, 36), (90, 150), denoise_model=den, denoise_rate=0.5)
    for fi in range(3):
        want = svc.upscale_single(frames[fi].clone())
        got = glue.upscale_single(frames[fi].clone(), model, lr_shape=(20, 36), output_shape=(90, 150), denoise_model=den,
                                  denoise_rate=0.5, first_frame=fi == 0)
        _same_u8(got, want)
    # blur_ker / sharpen_ker weights
    assert torch.equal(ns["blur_ker"](kernel_size=17, sigma=8.0).weight.data, glue.blur_weight(17, 8.0))
    assert torch.allclose(ns["sharpen_ker"](strength=0.00007).weight.data, glue.sharpen_weight(0.00007), atol=0, rtol=0)


@needs_ref
def test_srvgg_matches_live_reference():
    fac = ri.load_realesrgan_factory()
    torch.manual_seed(7)
    ref = fac.SRVGGNetCompact(3, 3, 64, 16, 4, "prelu").eval()
    mine = srvgg.SRVGGNetCompact(3, 3, 64, 16, 4).eval()
    mine.load_state_dict(ref.state_dict(), strict=True)
    x = torch.rand(2, 3, 9, 11)
    with torch.no_grad():
        assert (mine(x) - ref(x)).abs().max().item() == 0.0


@needs_ref
def test_bsvd_matches_live_reference():
    bm = ri.load_bsvd_model()
    with ri.cpu_shims():
        torch.manual_seed(11)
        ref = bm.BSVD(chns=[32, 64, 128], mid_ch=32, shift_input=False, norm="none", interm_ch=30, act="relu6",
                      pretrain_ckpt=None).eval()
        x = torch.rand(1, 6, 4, 16, 16)
        with torch.no_grad():
            want = ref(x)
            again = ref(x)  # state reset after every call (model.py:579)
    assert torch.equal(want, again)
    sd = bsvd.build_bsvd32(11)
    for k, v in ref.state_dict().items():
        assert torch.equal(sd[k], v), k
    got = bsvd.bsvd_forward(sd, x)
    assert (got - want).abs().max().item() <= 2e-5 * want.abs().max().item()


def test_colour_oracle_known_answers():
    """oracle/colour.py (BT.709 limited range): black / white / primaries land on the standard code values and the
    decode of the encode returns the colour within 4:2:0 rounding."""
    import numpy as np
    from oracle import colour
    cases = {(0, 0, 0): (16, 128, 128), (255, 255, 255): (235, 128, 128), (255, 0, 0): (63, 102, 240),
             (0, 255, 0): (173, 42, 26), (0, 0, 255): (32, 240, 118)}
    for rgb, yuv in cases.items():
        a = np.array(rgb, dtype=np.uint8).reshape(1, 1, 1, 3).repeat(2, 1).repeat(4, 2)
        q = colour.rgb_to_nv12(a)
        assert (int(q[0, 0]), int(q[0, 8]), int(q[0, 9])) == yuv, (rgb, q[0, 0], q[0, 8], q[0, 9])
        back = colour.nv12_to_rgb(q, 2, 4)[0, :, 0, 0] * 255
        assert np.abs(back - np.array(rgb)).max() <= 1.5
