"""FsrcnnUpscalerService(out_fmt=FMT_NV12) on every path: the NV12 frames must equal Engine.rgb_to_nv12 of the uint8 RGB
frames a service with the same settings returns, bit for bit and shape included."""
import os

import numpy as np
import pytest
import torch

from ss4k_b200 import _lib as L
from ss4k_b200 import multi_gpu, service
from oracle import bsvd, rrdbnet, srvgg
from tests.test_glue_gpu import GOLD, _golden_module

pytestmark = pytest.mark.gpu


def _frames(n, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(n, h // 8 + 1, w // 8 + 1, 3, generator=g)
    up = torch.nn.functional.interpolate(base.permute(0, 3, 1, 2), size=(h, w), mode="bilinear").permute(0, 2, 3, 1)
    return (up * 255 + torch.randn(n, h, w, 3, generator=g) * 6).clamp(0, 255).to(torch.uint8)


def _pair(output_shape, **kw):
    """(uint8 RGB service, NV12 service) with the same settings, both initialised."""
    out = []
    for fmt in (L.FMT_U8_NHWC, L.FMT_NV12):
        svc = service.FsrcnnUpscalerService(device=0, out_fmt=fmt, **kw)
        svc.proc_init()
        svc.output_shape = output_shape
        out.append(svc)
    return out


def _assert_nv12_of(engine, nv, rgb):
    """nv == rgb_to_nv12(rgb) with the packed-frame shape [..., h*3/2, w]."""
    lead, (h, w) = rgb.shape[:-3], rgb.shape[-3:-1]
    assert nv.dtype == torch.uint8 and tuple(nv.shape) == tuple(lead) + (h * 3 // 2, w), (nv.shape, rgb.shape)
    want = engine.rgb_to_nv12(rgb.reshape(-1, h, w, 3).contiguous()).view(nv.shape)
    assert torch.equal(nv, want)


def _srvgg_sd():
    torch.manual_seed(0)
    return srvgg.SRVGGNetCompact(3, 3, 64, 16, 4).eval().state_dict()


def _rrdb_sd(blocks=2):
    torch.manual_seed(0)
    return rrdbnet.RRDBNet(3, 3, 2, 64, blocks, 32).eval().state_dict()


@pytest.mark.parametrize("out_shape", [(180, 320), (100, 200), (400, 700), None])
def test_upscale_multi_srvgg_x4(engine, out_shape):
    """Net output 360 x 640: fused finalise + bicubic (factor 2), the two-pass resize (3.6 / 3.2), upscaling, no resize."""
    rgb_svc, nv_svc = _pair(out_shape, lr_level=3, denoising=False, model_name='realesr-animevideov3', state_dict=_srvgg_sd(),
                            batch_size=2)
    frames = _frames(2, 90, 160, 5).cuda()
    _assert_nv12_of(engine, nv_svc.upscale(frames), rgb_svc.upscale(frames))


@pytest.mark.parametrize("out_shape", [None, (150, 268)])
def test_upscale_multi_rrdb_x2(engine, out_shape):
    rgb_svc, nv_svc = _pair(out_shape, lr_level=3, denoising=False, model_name='RealESRGAN_x2plus', state_dict=_rrdb_sd(),
                            batch_size=2)
    frames = _frames(2, 96, 160, 1).cuda()
    _assert_nv12_of(engine, nv_svc.upscale(frames), rgb_svc.upscale(frames))


@pytest.mark.parametrize("denoising,out_shape", [(True, (720, 1280)), (False, (540, 960))])
def test_upscale_single(engine, denoising, out_shape):
    rgb_svc, nv_svc = _pair(out_shape, lr_level=0, denoising=denoising, denoise_rate=0.75, model_name='RealESRGAN_x2plus',
                            state_dict=_rrdb_sd(), denoise_state_dict=bsvd.build_bsvd32(0, weight_scale=0.5), single_mode=True)
    frames = _frames(2, 360, 640, 3).cuda()
    _assert_nv12_of(engine, nv_svc.upscale(frames), rgb_svc.upscale(frames))   # first frame, then the steady-state noise map


def test_upscale_temporal(engine):
    """18 frames through BSVD's ring buffers in jobs of 4, then flush(): the same entries in both formats, the frame-less
    entries of the filling delay line shaped [0, oh*3/2, ow]."""
    rgb_svc, nv_svc = _pair((720, 1280), lr_level=0, denoising=True, denoise_rate=0.75, batch_size=4,
                            model_name='RealESRGAN_x2plus', state_dict=_rrdb_sd(1),
                            denoise_state_dict=bsvd.build_bsvd32(0, weight_scale=0.5), single_mode=True, temporal_denoise=True)
    frames = _frames(18, 360, 640, 9)
    jobs = [frames[4 * k: 4 * k + 4] for k in range(5)]
    got = {}
    for name, svc in (("rgb", rgb_svc), ("nv", nv_svc)):
        entries = [svc.proc_job_recieved(service.UpscalerQueueEntry(frames=fr.cuda(), step=k)) for k, fr in enumerate(jobs)]
        entries += svc.flush()
        got[name] = entries
        svc.proc_cleanup()
    assert [e.step for e in got["nv"]] == [e.step for e in got["rgb"]]
    for e in got["nv"][:4]:   # 16 frames of latency
        assert e.step == -1 and tuple(e.frames.shape) == (0, 1080, 1280)
    done = [(a, b) for a, b in zip(got["rgb"], got["nv"]) if a.frames.shape[0]]
    assert sum(a.frames.shape[0] for a, _ in done) == 18
    for a, b in done:
        _assert_nv12_of(engine, b.frames, a.frames)


@pytest.fixture(scope="module")
def golden_pair(engine):
    """Both formats of FsrcnnUpscalerService with the stand-in nets the golden glue outputs were made with."""
    mg = _golden_module()
    model, den = mg.glue_models()
    out = []
    for fmt in (L.FMT_U8_NHWC, L.FMT_NV12):
        svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, model_name='realesr-animevideov3',
                                            state_dict=_srvgg_sd(), batch_size=2, out_fmt=fmt)
        svc.proc_init()
        svc.model = model
        svc._run_model = lambda lr: model(lr.permute(0, 3, 1, 2) / 255.0 if lr.dtype == torch.uint8 else lr).contiguous()
        out.append(svc)
    return out, mg, den


def test_golden_cases(engine, golden_pair):
    (rgb_svc, nv_svc), mg, den = golden_pair
    frames = torch.from_numpy(np.load(os.path.join(GOLD, "glue.npz"))["frames"]).cuda()
    for lr_shape, out_shape in mg.GLUE_MULTI_CASES:
        for svc in (rgb_svc, nv_svc):
            svc.single_mode, svc.denoising, svc.denoise_model = False, False, None
            svc.lr_shape, svc.output_shape = tuple(lr_shape), out_shape
        _assert_nv12_of(engine, nv_svc.upscale(frames), rgb_svc.upscale(frames))
    for use_den in (False, True):
        for svc in (rgb_svc, nv_svc):
            svc.single_mode, svc.denoise_rate = True, 0.75
            svc.lr_shape, svc.output_shape = tuple(mg.GLUE_SINGLE_LR), mg.GLUE_SINGLE_OUT
            svc.denoising, svc.denoise_model, svc.lr_prev = use_den, den if use_den else None, None
        for fi in range(2):
            _assert_nv12_of(engine, nv_svc.upscale(frames[fi:fi + 1]), rgb_svc.upscale(frames[fi:fi + 1]))


@pytest.mark.parametrize("out_shape", [(181, 320), (180, 322)])
def test_output_shape_nv12_cannot_hold_raises(engine, out_shape):
    svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, model_name='realesr-animevideov3',
                                        state_dict=_srvgg_sd(), out_fmt=L.FMT_NV12)
    svc.proc_init()
    svc.output_shape = out_shape
    with pytest.raises(L.Ss4kError, match="NV12"):
        svc.upscale(_frames(1, 90, 160, 2).cuda())
    svc.output_shape = (180, 320)   # the service still serves a size NV12 holds
    assert tuple(svc.upscale(_frames(1, 90, 160, 2).cuda()).shape) == (1, 270, 320)


def test_multi_gpu_front_returns_nv12(engine):
    """Two workers (both on cuda:0 when the box has one GPU) with out_fmt=FMT_NV12: the frames of the in-process service."""
    sd = {k: v.clone() for k, v in _srvgg_sd().items()}
    kw = dict(lr_level=0, denoising=False, model_name='realesr-animevideov3', state_dict=sd, out_fmt=L.FMT_NV12)
    one = service.FsrcnnUpscalerService(device=0, **kw)
    one.proc_init()
    g = torch.Generator().manual_seed(3)
    jobs = [torch.randint(0, 256, (2, 36, 64, 3), dtype=torch.uint8, generator=g) for _ in range(4)]
    want = [one.upscale(f.cuda()).cpu() for f in jobs]
    assert tuple(want[0].shape) == (2, 216, 256)
    front = multi_gpu.MultiGpuUpscalerService(devices=[0, 1 % torch.cuda.device_count()], **kw)
    front.start(ready_timeout=600)
    try:
        for i, f in enumerate(jobs):
            front.push_job(service.UpscalerQueueEntry(frames=f.cuda(), step=i, audio_segment=torch.zeros(1)))
        got = [front.get_result(timeout=120) for _ in jobs]
    finally:
        front.stop()
    assert [e.step for e in got] == list(range(len(jobs)))
    for e, w in zip(got, want):
        assert torch.equal(e.frames.cpu(), w)
