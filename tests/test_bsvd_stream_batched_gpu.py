"""BSVD ring-buffer streams that take several frames per push (ss4k_bsvd_stream_push_frames): each conv runs once over
the pushed frames, its ring slots wrapping inside the kernel.  Pushed in batches, a stream must give the bits of the
same frames pushed one at a time, and match the clip program as the one-frame streams do."""
import ctypes

import pytest
import torch

from ss4k_b200 import _lib as L
from ss4k_b200 import bsvd as native_bsvd
from ss4k_b200 import service
from oracle import bsvd, rrdbnet

pytestmark = pytest.mark.gpu

H, W = 32, 136
SIZES = [1, 3, 4, 2, 4, 4, 1, 2, 3, 4, 4, 4, 1, 1, 3, 2, 4, 3, 4, 4, 2, 4]   # 70 frames: every ring wraps at least twice


def _pieces(t, sizes=SIZES):
    out, i, k = [], 0, 0
    while i < t:
        n = min(sizes[k % len(sizes)], t - i)
        out.append((i, i + n))
        i, k = i + n, k + 1
    return out


def _frames(t, fmt, seed):
    g = torch.Generator().manual_seed(seed)
    if fmt == L.FMT_NV12:
        return torch.randint(16, 236, (t, H * 3 // 2, W), generator=g, dtype=torch.uint8).cuda()
    if fmt == L.FMT_U8_NHWC:
        return torch.randint(0, 256, (t, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    x = torch.rand(t, 4, H, W, generator=g)
    x[:, 3] = 0.075
    return x.cuda()


def _one_at_a_time(model, frames, fmt):
    s = model.stream(H, W, in_fmt=fmt, noise=0.075)
    outs = [o for o in (s.push(frames[i]) for i in range(frames.shape[0])) if o is not None] + list(s.flush())
    s.close()
    return torch.cat(outs, dim=0)


def _batched(model, frames, fmt, max_frames=4, engine=None, steady_launches=None):
    s = model.stream(H, W, in_fmt=fmt, noise=0.075, max_frames=max_frames)
    t, outs, pushed = frames.shape[0], [], 0
    for i0, i1 in _pieces(t):
        before = engine.launch_count if engine is not None else 0
        o = s.push_frames(frames[i0:i1])
        pushed += i1 - i0
        # frames t-16 .. t+n-17 that exist, oldest first
        assert o.shape[0] == max(0, pushed - 16) - max(0, i0 - 16)
        if engine is not None and i0 > 16:
            steady_launches.setdefault(i1 - i0, set()).add(engine.launch_count - before)
        outs.append(o)
    outs += list(s.flush())
    s.close()
    return torch.cat(outs, dim=0)


def _model(split):
    sd = bsvd.build_bsvd32(0, weight_scale=1.0 if split else 0.5)
    return native_bsvd.NativeBSVD(sd, device=0, act_mode=L.ACT_F16_SPLIT if split else L.ACT_F16)


@pytest.mark.parametrize("split", [False, True])
def test_push_sizes_equal_single_pushes_and_clip(engine, split):
    """70 frames pushed as 1, 3, 4, 2, 4, ... frames per call == the same frames pushed one at a time, bit for bit, and
    == the clip program (split precision: bit for bit, fp16: within the one-frame streams' 1e-3)."""
    model = _model(split)
    x = _frames(70, L.FMT_F32_NCHW, 31)
    one = _one_at_a_time(model, x, L.FMT_F32_NCHW)
    got = _batched(model, x, L.FMT_F32_NCHW)
    assert tuple(got.shape) == (70, 3, H, W)
    assert torch.equal(got, one)
    clip = model(x.unsqueeze(0))[0]
    if split:
        assert torch.equal(got, clip)
    else:
        assert (got - clip).abs().max().item() <= 1e-3


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("fmt", [L.FMT_U8_NHWC, L.FMT_NV12])
@pytest.mark.parametrize("split", [False, True])
def test_frame_formats_and_graphs(engine, monkeypatch, split, fmt, graph):
    """uint8 RGB / NV12 frames, graphed steady-state pushes and per-layer launches (SS4K_NO_STREAM_GRAPH=1): batched ==
    one at a time bit for bit.  A steady-state push of n frames issues as many launches as a one-frame push (graphed
    pushes count the launches of their captured graph): each conv runs once per push, the layout step once more where
    the ring wraps."""
    if not graph:
        monkeypatch.setenv("SS4K_NO_STREAM_GRAPH", "1")
    model = _model(split)
    x = _frames(70, fmt, 41)
    one = _one_at_a_time(model, x, fmt)
    launches = {}
    got = _batched(model, x, fmt, engine=engine, steady_launches=launches)
    assert torch.equal(got, one)
    assert set(launches) == {1, 2, 3, 4}
    one_frame = min(launches[1])
    for n in (1, 2, 3, 4):   # each conv once per push; the layout step takes a second launch where the ring wraps
        assert min(launches[n]) >= one_frame and max(launches[n]) <= one_frame + 1, (n, launches)


@pytest.mark.parametrize("split", [False, True])
def test_short_clip_one_batch_then_reset(engine, split):
    """A clip shorter than 16 frames pushed as one batch comes out of the flush alone; after reset a second clip sees
    nothing of the first."""
    model = _model(split)
    s = model.stream(H, W, max_frames=8)
    x1, x2 = _frames(7, L.FMT_F32_NCHW, 51), _frames(5, L.FMT_F32_NCHW, 52)
    assert s.push_frames(x1).shape[0] == 0
    got1 = torch.cat(list(s.flush()), dim=0)
    s.reset()
    assert s.push_frames(x2).shape[0] == 0
    got2 = torch.cat(list(s.flush()), dim=0)
    s.close()
    assert torch.equal(got1, _one_at_a_time(model, x1, L.FMT_F32_NCHW))
    assert torch.equal(got2, _one_at_a_time(model, x2, L.FMT_F32_NCHW))
    clip2 = model(x2.unsqueeze(0))[0]
    assert (got2 - clip2).abs().max().item() <= (0.0 if split else 1e-3)


def test_rejected_arguments(engine):
    """n = 0, n > max_frames and a push after flush (without reset) fail with SS4K_E_INVALID."""
    model = _model(False)
    s = model.stream(H, W, max_frames=3)
    x = _frames(4, L.FMT_F32_NCHW, 61)
    out = torch.empty(4, 3, H, W, device="cuda")
    got = ctypes.c_int(0)
    for n in (0, 4, -1):
        rc = s.lib.ss4k_bsvd_stream_push_frames(s.hdl, ctypes.c_void_p(x.data_ptr()), n, ctypes.c_void_p(out.data_ptr()),
                                                ctypes.byref(got), None)
        assert rc != L.OK
    with pytest.raises(L.Ss4kError):
        s.push_frames(x)
    assert s.push_frames(x[:3]).shape[0] == 0
    list(s.flush())
    with pytest.raises(L.Ss4kError):
        s.push_frames(x[:1])
    with pytest.raises(L.Ss4kError):
        s.push(x[0])
    s.reset()
    assert s.push_frames(x[:2]).shape[0] == 0
    s.close()


def test_service_jobs_of_four_equal_jobs_of_one(engine):
    """temporal_denoise=True: jobs of 4 frames (one push each) return the frames, step and audio order of jobs of one
    frame, bit for bit."""
    torch.manual_seed(0)
    net = rrdbnet.RRDBNet(3, 3, 2, 64, 1, 32).eval()
    sd = bsvd.build_bsvd32(0, weight_scale=0.5)
    t, lh, lw = 22, 360, 640          # lr_level 0: the area resize is the identity
    g = torch.Generator().manual_seed(9)
    frames = torch.randint(0, 256, (t, lh, lw, 3), generator=g, dtype=torch.uint8)

    def run(job):
        svc = service.FsrcnnUpscalerService(lr_level=0, device=0, denoising=True, denoise_rate=0.75, batch_size=4,
                                            model_name='RealESRGAN_x2plus', state_dict=net.state_dict(),
                                            denoise_state_dict=sd, single_mode=True, temporal_denoise=True)
        assert tuple(svc.lr_shape) == (lh, lw)
        svc.proc_init()
        svc.output_shape = (2 * lh, 2 * lw)
        entries = []
        for k in range((t + job - 1) // job):
            fr = frames[job * k: job * k + job]
            entries.append(svc.proc_job_recieved(service.UpscalerQueueEntry(frames=fr.cuda(), step=100 + k,
                                                                            audio_segment=("audio", k))))
        entries += svc.flush()
        svc.proc_cleanup()
        done = [e for e in entries if e.frames.shape[0]]
        return done

    four, one = run(4), run(1)
    assert [e.step for e in four] == [100 + k for k in range((t + 3) // 4)]
    assert [e.audio_segment for e in four] == [("audio", k) for k in range((t + 3) // 4)]
    assert [e.step for e in one] == [100 + k for k in range(t)]
    a, b = torch.cat([e.frames for e in four], dim=0), torch.cat([e.frames for e in one], dim=0)
    assert a.shape[0] == t and torch.equal(a, b)
