"""NV12 output of RRDBNet plans on the GPU.  The defined result is ss4k_rgb_to_nv12 applied to the same plan's uint8 RGB
output, bit for bit: every case runs a U8 plan and an NV12 plan of the same net on the same input, converts the U8
frames with Engine.rgb_to_nv12 and compares every byte.  The NV12 output buffer sits at the front of a larger
allocation filled with a canary byte: nothing past the frames may change."""
import pytest
import torch

from ss4k_b200 import _lib as L
from ss4k_b200 import realesrgan
from oracle import rrdbnet

pytestmark = pytest.mark.gpu

CANARY = 0xA5
TAIL = 4096


def _net(scale, blocks, seed=0):
    """Seeded RRDBNet with non-zero biases and a conv_last that spreads the output over [0, 1] (and past both ends, so
    clamping takes part): a random-init net otherwise leaves most bytes at one value."""
    torch.manual_seed(seed)
    net = rrdbnet.RRDBNet(3, 3, scale, 64, blocks, 32).eval()
    with torch.no_grad():
        for p in net.parameters():
            if p.ndim == 1:
                torch.nn.init.uniform_(p, -0.1, 0.1)
        net.conv_last.weight.mul_(8.0)
        net.conv_last.bias.fill_(0.5)
    return net


def _canary_out(plan):
    shape = plan.out_shape()
    nbytes = torch.Size(shape).numel()
    assert nbytes == plan.out_bytes
    buf = torch.full((nbytes + TAIL,), CANARY, dtype=torch.uint8, device="cuda")
    return buf, buf[:nbytes].view(shape)


def _check_nv12(engine, u8, nv12, buf):
    """u8: [n, H, W, 3] uint8 frames of the U8 plan; nv12: the NV12 plan's [n, H*3/2, W] output inside `buf`."""
    n, H, W, _ = u8.shape
    assert tuple(nv12.shape) == (n, H * 3 // 2, W) and nv12.dtype == torch.uint8
    want = engine.rgb_to_nv12(u8.contiguous())
    torch.cuda.synchronize()
    assert len(torch.unique(u8)) > 64, "degenerate test image"
    got = nv12.reshape(n, -1)
    bad = (got != want).nonzero()
    assert bad.numel() == 0, f"{bad.shape[0]} bytes differ, first at {bad[0].tolist()}"
    assert bool((buf[nv12.numel():] == CANARY).all()), "bytes past the NV12 frames were written"


# output widths that are and are not multiples of 128; row counts whose plain even split over the grid gives some CTA an
# odd first row (tests/test_nv12_out_cpu.py)
CASES = [(s, n, h, w) for s in (2, 4) for n in (1, 3) for (h, w) in ((96, 128), (70, 46))] + \
        [(2, 1, 720, 1280), (2, 3, 720, 1280), (4, 1, 720, 1280)]


@pytest.mark.parametrize("scale,n,h,w", CASES)
def test_rrdb2_nv12_equals_u8_then_rgb_to_nv12(engine, scale, n, h, w):
    net = _net(scale, 2, seed=scale * 100 + n)
    model = realesrgan.NativeRRDBNet(net.state_dict(), scale=scale, num_block=2, device=0)
    x = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(n * 7 + h)).cuda()
    pu = model._plan(n, h, w, L.FMT_F32_NCHW, L.FMT_U8_NHWC)
    pn = model._plan(n, h, w, L.FMT_F32_NCHW, L.FMT_NV12)
    assert pn.out_nchw == pu.out_nchw == (n, 3, h * scale, w * scale)
    assert pn.out_bytes * 2 == pu.out_bytes
    assert pn.launches == pu.launches and pn.steps == pu.steps    # the conversion is inside the last conv
    u8 = pu.run(x)
    buf, out = _canary_out(pn)
    pn.run(x, out)
    _check_nv12(engine, u8, out, buf)
    # per-step profile: same steps as the U8 plan, the last one the streaming conv
    prof = pn.profile(x, out)
    assert len(prof) == pn.steps and prof[-1][2] == 1
    _check_nv12(engine, u8, out, buf)


def test_rrdb23_x2_720p_graph_on_off_deterministic(engine):
    net = _net(2, 23, seed=23)
    x = torch.rand(1, 3, 720, 1280, generator=torch.Generator().manual_seed(5)).cuda()
    u8 = None
    for use_graph in (True, False):
        model = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=23, device=0, use_graph=use_graph)
        if u8 is None:
            pu = model._plan(1, 720, 1280, L.FMT_F32_NCHW, L.FMT_U8_NHWC)
            u8 = pu.run(x).clone()
            pu.close()
        pn = model._plan(1, 720, 1280, L.FMT_F32_NCHW, L.FMT_NV12)
        assert (pn.graph_steps > 0) == use_graph
        first = None
        for _ in range(2):
            buf, out = _canary_out(pn)
            pn.run(x, out)
            _check_nv12(engine, u8, out, buf)
            if first is not None:
                assert torch.equal(out, first)
            first = out.clone()
        pn.close()


def test_tiled_1080p_tile512_nv12_two_step(engine):
    """Tiled plan (1920x1080, tile 512, pad 10): the tile classes paste uint8 RGB into a frame of the plan and one
    conversion writes the caller's NV12 buffer."""
    net = _net(2, 2, seed=11)
    model = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=2, device=0, tile=512, tile_pad=10)
    x = torch.rand(1, 3, 1080, 1920, generator=torch.Generator().manual_seed(6)).cuda()
    pu = model._plan(1, 1080, 1920, L.FMT_F32_NCHW, L.FMT_U8_NHWC)
    pn = model._plan(1, 1080, 1920, L.FMT_F32_NCHW, L.FMT_NV12)
    assert pn.launches == pu.launches + 1
    u8 = pu.run(x)
    buf, out = _canary_out(pn)
    pn.run(x, out)
    _check_nv12(engine, u8, out, buf)
    # host path: the plan's NV12 byte count crosses the copy
    out_host = torch.empty(pn.out_shape(), dtype=torch.uint8).pin_memory()
    pn.run_host(x.cpu().pin_memory(), out_host)
    assert torch.equal(out_host, out.cpu())


def test_last_conv_off_the_streaming_kernel_takes_two_steps(engine, monkeypatch):
    """SS4K_NO_STREAM=1 puts every conv on the tile kernel: the last conv writes uint8 RGB into the plan's frame and a
    conversion step of its own (listed by the profile as a colour kernel) writes NV12."""
    monkeypatch.setenv("SS4K_NO_STREAM", "1")
    net = _net(2, 1, seed=12)
    model = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=1, device=0)
    x = torch.rand(2, 3, 48, 70, generator=torch.Generator().manual_seed(7)).cuda()
    pu = model._plan(2, 48, 70, L.FMT_F32_NCHW, L.FMT_U8_NHWC)
    pn = model._plan(2, 48, 70, L.FMT_F32_NCHW, L.FMT_NV12)
    assert pn.steps == pu.steps + 1 and pn.launches == pu.launches + 1
    u8 = pu.run(x)
    buf, out = _canary_out(pn)
    pn.run(x, out)
    _check_nv12(engine, u8, out, buf)
    prof = pn.profile(x, out)
    assert len(prof) == pn.steps and prof[-1][2] == 0 and prof[-2][2] == 2
    _check_nv12(engine, u8, out, buf)


def test_pipeline_nv12_out_equals_u8_pipeline_then_rgb_to_nv12(engine):
    """DenoiseUpscalePipeline with out_fmt = NV12 on a short NV12 720p chunk with an owned sub-range, on the device path
    and on the pinned host path."""
    from ss4k_b200 import bsvd as nb
    from ss4k_b200.pipeline import DenoiseUpscalePipeline
    from oracle import bsvd, colour
    h, w, T, own = 720, 1280, 5, slice(1, 4)
    rgb8 = torch.randint(0, 256, (T, h // 8, w // 8, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(9))
    rgb8 = torch.nn.functional.interpolate(rgb8.permute(0, 3, 1, 2).float(), size=(h, w), mode="bilinear")
    rgb8 = rgb8.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().numpy()
    nv = torch.from_numpy(colour.rgb_to_nv12(rgb8)).reshape(T, -1).contiguous()
    den = nb.NativeBSVD(bsvd.build_bsvd32(0), device=0, act_mode="auto", out_dtype=torch.float16)
    sr = realesrgan.NativeRRDBNet(_net(2, 2, seed=13).state_dict(), scale=2, num_block=2, device=0)
    pu = DenoiseUpscalePipeline(den, sr, h, w, 0.075, nv12=True, out_fmt=L.FMT_U8_NHWC)
    pn = DenoiseUpscalePipeline(den, sr, h, w, 0.075, nv12=True, out_fmt=L.FMT_NV12)
    assert pn.out_frame_shape() == (2 * h * 3 // 2, 2 * w)
    frames = nv.cuda()
    u8 = pu.run(frames, own)
    got = pn.run(frames, own)
    assert got.dtype == torch.uint8 and tuple(got.shape) == (3, 2 * h * 3 // 2, 2 * w)
    want = engine.rgb_to_nv12(u8)
    torch.cuda.synchronize()
    assert len(torch.unique(u8)) > 64
    assert torch.equal(got.reshape(3, -1), want)
    out_host = torch.empty((3,) + pn.out_frame_shape(), dtype=torch.uint8).pin_memory()
    pn.run_host(nv.pin_memory(), own, out_host)
    pn.host_sync()
    assert torch.equal(out_host.reshape(3, -1), want.cpu())
