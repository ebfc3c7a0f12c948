"""BASELINE.json's full sizes (configs[1]: RRDBNet-23 x2, 1280x720 -> 2560x1440) on the GPU:
  * parity against the CPU oracle on the WHOLE frame (one frame: the fp32 oracle needs ~0.5 minute of host time)
  * size-independent properties that need no oracle: batch invariance (a frame's result does not depend on its
    batch neighbours, bit for bit), determinism, and translation equivariance of the interior (the net is a stack of
    zero-padded 3x3 convs behind a pixel-unshuffle(2): shifting the input by an even number of pixels shifts the
    output by twice that, away from the borders) -- this moves every feature across the kernel's strip / band /
    accumulator-ring boundaries, which sit at fixed image positions."""
import math
import os

import pytest
import torch

from ss4k_b200 import _lib as L
from ss4k_b200 import realesrgan
from oracle import rrdbnet

pytestmark = pytest.mark.gpu

H, W = 720, 1280


@pytest.fixture(scope="module")
def net():
    torch.manual_seed(0)
    return rrdbnet.RRDBNet(3, 3, 2, 64, 23, 32).eval()


@pytest.fixture(scope="module")
def model(engine, net):
    return realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=23, device=0)


def _frames(n, seed=1234):
    g = torch.Generator().manual_seed(seed)
    # smooth content + noise: random-init RRDBNet amplifies pure noise less informatively
    base = torch.rand(n, 3, H // 8, W // 8, generator=g)
    x = torch.nn.functional.interpolate(base, size=(H, W), mode="bilinear", align_corners=False)
    return (x + 0.05 * torch.randn(n, 3, H, W, generator=g)).clamp(0, 1)


@pytest.fixture(scope="module")
def full_frame(net):
    x = _frames(1)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        want = net(x).clamp(0, 1)
    return x, want


def _gate(got, want):
    mse = torch.mean((got - want) ** 2).item()
    psnr = 99.0 if mse == 0 else -10 * math.log10(mse)
    return psnr, (got - want).abs().max().item() * 255


def test_rrdbnet_x2_720p_full_frame_vs_oracle(model, full_frame):
    x, want = full_frame
    got = model(x.cuda()).float().cpu().clamp(0, 1)
    assert tuple(got.shape) == (1, 3, 2 * H, 2 * W)
    psnr, maxabs = _gate(got, want)
    print(f"RRDBNet-23 x2 1280x720 full frame (fp16 operands): PSNR {psnr:.1f} dB, max|err| {maxabs:.3f}/255")
    assert psnr >= 50 and maxabs <= 2.0


def test_rrdbnet_x2_720p_bf16_report(engine, net, full_frame):
    """BASELINE.json configs[1] says "bf16": run it at net level on the whole frame and REPORT it.  SURVEY.md H2 predicts
    that bf16 operands miss the max-abs gate on RRDBNet (8 mantissa bits through 351 convs) -- which is why fp16 is the
    engine's default; the test is an expected failure whose message carries the measured numbers."""
    x, want = full_frame
    m16 = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=23, device=0, act_mode=L.ACT_BF16)
    got = m16(x.cuda()).float().cpu().clamp(0, 1)
    m16.close()
    psnr, maxabs = _gate(got, want)
    msg = f"RRDBNet-23 x2 1280x720 full frame (bf16 operands): PSNR {psnr:.1f} dB, max|err| {maxabs:.3f}/255"
    print(msg)
    assert psnr >= 40, msg          # a broken bf16 path is a failure, a precision miss is the expected outcome
    if not (psnr >= 50 and maxabs <= 2.0):
        pytest.xfail(msg + " -- bf16 misses the north-star gate as predicted (SURVEY.md H2); fp16 is the default")


def test_batch_invariance_and_determinism(model):
    x = _frames(3, seed=7).cuda()
    plan3 = model._plan(3, H, W, L.FMT_F32_NCHW, L.FMT_F16_NCHW)
    plan1 = model._plan(1, H, W, L.FMT_F32_NCHW, L.FMT_F16_NCHW)
    assert plan1.launches == plan1.steps and plan3.launches == plan3.steps   # one kernel launch per step
    a = plan3.run(x).clone()
    b = plan3.run(x).clone()
    assert torch.equal(a, b)
    for i in range(3):
        assert torch.equal(plan1.run(x[i:i + 1].contiguous()), a[i:i + 1])


@pytest.mark.parametrize("dy,dx", [(2, 0), (0, 2), (6, 130), (14, 4)])
def test_translation_equivariance_of_the_interior(model, dy, dx):
    """out(shift(x))[interior] ~= shift(out(x))[interior].  The arithmetic of a pixel does not depend on its position
    (same K order per pixel whatever strip / band / accumulator slot it lands in), so the only difference between the two
    runs is the zero padding that moved with the shift: the receptive field (about 350 trunk pixels) is larger than the
    256-pixel margin, but border influence decays fast through the 0.2-scaled residual blocks.  Asserted: the interior
    agrees within the north-star tolerance (2/255); a strip- or band-boundary bug shows up as an O(1) difference."""
    x = _frames(1, seed=3).cuda()
    plan = model._plan(1, H, W, L.FMT_F32_NCHW, L.FMT_F16_NCHW)
    ref = plan.run(x).clone()
    xs = torch.zeros_like(x)
    xs[:, :, dy:, dx:] = x[:, :, :H - dy, :W - dx]
    out = plan.run(xs)
    # the zero padding moved by (dy, dx): compare far from every border (receptive field ~ 2*(1+23*15+1)+... px at
    # trunk scale is larger than the frame, but border effects decay: use a tolerance instead of an exact margin)
    m = 256
    a = out[:, :, 2 * dy + m:2 * H - m, 2 * dx + m:2 * W - m].float()
    b = ref[:, :, m:2 * (H - dy) - m, m:2 * (W - dx) - m].float()
    assert a.shape == b.shape
    diff = (a - b).abs().max().item()
    print(f"shift ({dy},{dx}): interior max |diff| {diff:.2e}")
    assert diff <= 2.0 / 255


def test_run_host_async_matches_run_host(engine):
    """The pipelined host path (ss4k_run_host_async: H2D, kernels and D2H of neighbouring frames overlap on three
    streams, two staging slots) returns bit for bit what the serial ss4k_run_host returns, frame by frame."""
    import torch
    from ss4k_b200 import _lib as L, realesrgan
    from oracle import rrdbnet
    torch.manual_seed(5)
    net = rrdbnet.RRDBNet(3, 3, 2, 64, 2, 32).eval()
    model = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=2, device=0)
    plan = model._plan(1, 96, 160, L.FMT_U8_NHWC, L.FMT_U8_NHWC)
    frames = [torch.randint(0, 256, (1, 96, 160, 3), dtype=torch.uint8).pin_memory() for _ in range(5)]
    want = []
    for f in frames:
        o = torch.empty(1, 192, 320, 3, dtype=torch.uint8).pin_memory()
        plan.run_host(f, o)
        want.append(o.clone())
    outs = [torch.empty(1, 192, 320, 3, dtype=torch.uint8).pin_memory() for _ in range(5)]
    for f, o in zip(frames, outs):
        plan.run_host_async(f, o)
    plan.host_sync()
    for w, o in zip(want, outs):
        assert torch.equal(w, o)
    assert not torch.equal(want[0], want[1])


def test_early_activation_loads_are_sound(net, monkeypatch):
    """StreamParams::early_kb_mask (K blocks requested before griddepcontrol.wait) relies on one resident CTA per SM;
    the engine checks the occupancy when it sets the mask, and the result must not depend on it: conv-by-conv trunk
    with and without the early loads, bit for bit at full size (small shapes never take this path)."""
    x = _frames(1, seed=13).cuda()
    a = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=23, device=0)
    ya = a._plan(1, H, W, L.FMT_F32_NCHW, L.FMT_F16_NCHW).run(x).clone()
    monkeypatch.setenv("SS4K_NO_EARLY_LOAD", "1")
    b = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=23, device=0)
    yb = b._plan(1, H, W, L.FMT_F32_NCHW, L.FMT_F16_NCHW).run(x).clone()
    assert torch.equal(ya, yb)
    a.close()
    b.close()
