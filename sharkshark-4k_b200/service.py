"""Drop-in for the reference's upscaler service (outer boundary of the hot path).

Reference: src/upscale/fsrcnn_upscaler.py:86-326 ``FsrcnnUpscalerService`` (+ src/upscale/upscaler_base.py:17-63).
Same constructor keywords, same attributes (``lr_shape``, ``output_shape``, ``profiler``), same methods
(``proc_init``, ``proc_cleanup``, ``upscale``, ``upscale_multi``, ``upscale_single``, ``proc_job_recieved``):
``upscale(frames uint8 [N,H,W,3] on the device) -> uint8 [N,H',W',3]``, or with ``out_fmt=FMT_NV12`` packed NV12 frames
``uint8 [N,H'*3/2,W']`` (Y plane, then interleaved UV) that an encoder surface takes as they are (``ss4k_nv12_unpack``).  The queue / process plumbing of
``BaseService`` is NOT re-implemented: in the reference tree this class is mixed into ``BaseUpscalerService``
(see INTEGRATION.md); stand-alone it is driven by calling ``proc_init()`` then ``upscale()``.

All arithmetic runs in libss4k.so: the convnets (tcgen05 kernels) and the service glue (statistics, area
pooling, low-res gaussian, finalising pass, bicubic, sharpen: csrc/glue.cu).  torch is used for device buffers
and streams only.
"""
import collections
import ctypes
import math
import time
from dataclasses import dataclass

import torch

from . import _lib as L
from . import bsvd as native_bsvd
from . import realesrgan as native_esrgan
from .engine import Engine


@dataclass
class UpscalerQueueEntry:
    """src/upscale/upscaler_base.py:17-24"""
    frames: torch.Tensor = None
    audio_segment: torch.Tensor = None
    step: int = 0
    elapsed: float = 0
    last_modified: float = 0
    profiler: object = None


class _NullProfiler:
    """Stands in for src/util/profiler.py when the caller attaches none; keeps the region keys alive."""

    def start(self, name):
        pass

    def end(self, name):
        pass


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _fmt(t):
    if t.dtype == torch.uint8:
        return 2
    return 1 if t.dtype == torch.float16 else 0


def frame_shape(out_fmt, h, w):
    """Shape of one output frame of (h, w) pixels: (h, w, 3) for uint8 RGB, (h*3/2, w) for packed NV12.  NV12 needs an
    even height and a width divisible by 4; other sizes raise Ss4kError rather than yield a truncated frame."""
    if out_fmt == L.FMT_U8_NHWC:
        return (h, w, 3)
    if out_fmt == L.FMT_NV12:
        if h % 2 or w % 4:
            raise L.Ss4kError(f"NV12 output needs an even height and a width divisible by 4, not {h}x{w} "
                              "(set output_shape to such a size, or use out_fmt=FMT_U8_NHWC)")
        return (h * 3 // 2, w)
    raise ValueError(f"out_fmt must be FMT_U8_NHWC ({L.FMT_U8_NHWC}) or FMT_NV12 ({L.FMT_NV12}), not {out_fmt!r}")


def gaussian_kernel(kernel_size=3, sigma=0.5):
    """blur_ker weights (fsrcnn_upscaler.py:20-52): normalised 2-D gaussian."""
    ax = torch.arange(kernel_size, dtype=torch.float32) - (kernel_size - 1) / 2.0
    g = torch.exp(-(ax[:, None] ** 2 + ax[None, :] ** 2) / (2.0 * sigma ** 2)) / (2.0 * math.pi * sigma ** 2)
    return (g / g.sum()).contiguous()


# Frames per BSVD push in temporal mode: the orchestrator hands the service jobs of up to 4 frames, so a job is one push
# (each conv of the stream runs once over its frames instead of once per frame).
_TEMPORAL_PUSH = 4


class FsrcnnUpscalerService:
    LR_SHAPES = [(360, 640), (540, 960), (630, 1120), (720, 1280), (900, 1600), (1080, 1920)]  # :93-100

    def __init__(self, lr_level=3, device=0, on_queue=None, denoising=True, denoise_rate=1.0,
                 upscaler_model='realesrgan', batch_size=1, jit_mode=None, lr_hr_resize=True,
                 model_name=None, state_dict=None, denoise_state_dict=None, act_mode=L.ACT_F16,
                 denoise_act_mode="auto", single_mode=None, temporal_denoise=False, out_fmt=L.FMT_U8_NHWC):
        if out_fmt not in (L.FMT_U8_NHWC, L.FMT_NV12):
            raise ValueError(f"out_fmt must be FMT_U8_NHWC ({L.FMT_U8_NHWC}) or FMT_NV12 ({L.FMT_NV12}), not {out_fmt!r}")
        self.lr_shape = self.LR_SHAPES[lr_level]
        self.scale = 4
        self.denoise_rate = denoise_rate
        self.hr_shape = (1440, 2560)
        self.device = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        self.on_queue = on_queue
        self.output_shape = None
        self.upscaler_model = upscaler_model
        # :109 makes single_mode = (upscaler_model != 'realesrgan'), which only the FSRCNN model (out of scope here) can
        # reach; the keyword selects the per-frame denoise + upscale path (upscale_single) for the RealESRGAN models
        self.single_mode = (upscaler_model != 'realesrgan') if single_mode is None else bool(single_mode)
        self.denoising = denoising
        self.batch_size = batch_size
        self.jit_mode = jit_mode
        self.lr_hr_resize = lr_hr_resize
        self.profiler = _NullProfiler()
        # extensions (no network here: weights are handed in, not downloaded as in realesrgan/factory.py:140-150)
        self.model_name = model_name
        self.state_dict = state_dict
        self.denoise_state_dict = denoise_state_dict
        self.act_mode = act_mode
        self.denoise_act_mode = denoise_act_mode   # 'auto': fp16, or fp16 hi/lo split for kaiming-magnitude weights
        # temporal_denoise: upscale_single feeds BSVD's persistent ring buffers (BSVD.feedin_one_element, bsvd/model.py:
        # 510-513) instead of one F = 1 clip per frame (fsrcnn_upscaler.py:277): every frame is denoised with its +-16
        # temporal neighbours and leaves the service 16 frames late (jobs are delayed as a whole, see proc_job_recieved)
        self.temporal_denoise = bool(temporal_denoise)
        # out_fmt: frames leave as uint8 RGB [N,H,W,3] (the reference's) or as packed NV12 [N,H*3/2,W] for an encoder; the
        # colour-match finalising kernel writes NV12 itself, so no separate conversion pass runs
        self.out_fmt = out_fmt
        self.model = None

    # ------------------------------------------------------------------ life cycle (fsrcnn_upscaler.py:118-142)
    def proc_init(self):
        self.lr_prev = None
        self.lr_prev_diff_map = None
        if self.upscaler_model != 'realesrgan':
            raise Exception(self.upscaler_model)   # FSRCNN is out of scope of this engine (SURVEY.md section 2 row 10)
        args = native_esrgan.ArgsData()
        if self.model_name:
            args.model_name = self.model_name
        self.model = native_esrgan.build_model(factor=self.scale, device=self.device.index or 0, input_shape=self.lr_shape,
                                               batch_size=self.batch_size, denoise_rate=self.denoise_rate,
                                               jit_mode=self.jit_mode, args=args, state_dict=self.state_dict,
                                               act_mode=self.act_mode)
        self.model.out_dtype = torch.float16        # the reference's JitWrapper returns fp16 (factory.py:242-245)
        self.engine = Engine.get(self.device.index or 0)
        self.lib = self.engine.lib
        # only upscale_single uses the denoiser (fsrcnn_upscaler.py:245-284): the multi-frame default must not need a
        # BSVD checkpoint, so it is built here for single_mode and on first use otherwise
        self.denoise_model = None
        if self.denoising and self.single_mode:
            self._build_denoiser()
        self.match_blur = gaussian_kernel(8 * 2 + 1, 8.0).to(self.device)     # :138
        self._sums = {}
        self._den_stream = None      # temporal mode: the BSVD ring-buffer stream, the LR frames in flight, delayed jobs
        self._lr_fifo = collections.deque()
        self._jobs = collections.deque()
        self._ready = collections.deque()

    def _build_denoiser(self):
        self.denoise_model = native_bsvd.build_model(device=self.device.index or 0, input_shape=self.lr_shape,
                                                     state_dict=self.denoise_state_dict, act_mode=self.denoise_act_mode)

    def proc_cleanup(self):
        if self._den_stream is not None:
            self._den_stream.close()
            self._den_stream = None

    def proc_job_recieved(self, job):
        """src/upscale/upscaler_base.py:40-55"""
        self.profiler = job.profiler if job.profiler is not None else _NullProfiler()
        t = time.time()
        self.profiler.end('recoder.output')
        self.profiler.start('upscaler.upscale')
        frames_up = self.upscale(job.frames)
        self.profiler.end('upscaler.upscale')
        elapsed = time.time() - t
        self.profiler.start('upscaler.output')
        if self._temporal():
            # delay line of whole jobs: the entry returned for this job carries the frames, step and audio segment of the
            # oldest job whose frames have all left the 16-frame pipeline (an entry without frames while it fills)
            self._ready.extend(frames_up[i] for i in range(frames_up.shape[0]))
            self._jobs.append((job, job.frames.shape[0]))
            return self._pop_delayed(elapsed)
        return UpscalerQueueEntry(frames=frames_up, step=job.step, audio_segment=job.audio_segment, elapsed=elapsed,
                                  last_modified=time.time(), profiler=job.profiler)

    def _temporal(self):
        return self.temporal_denoise and self.denoising and self.single_mode

    def _pop_delayed(self, elapsed=0.0):
        if self._jobs and len(self._ready) >= self._jobs[0][1]:
            old, n = self._jobs.popleft()
            frames = torch.stack([self._ready.popleft() for _ in range(n)], dim=0)
            return UpscalerQueueEntry(frames=frames, step=old.step, audio_segment=old.audio_segment, elapsed=elapsed,
                                      last_modified=time.time(), profiler=old.profiler)
        return UpscalerQueueEntry(frames=self._no_frames(), step=-1,
                                  audio_segment=None, elapsed=elapsed, last_modified=time.time(), profiler=None)

    def _no_frames(self):
        """The frame-less result while the temporal pipeline fills: [0, *frame] of output_shape ((0, 0) while unset)."""
        oh, ow = self.output_shape if self.output_shape is not None else (0, 0)
        return torch.empty((0,) + frame_shape(self.out_fmt, oh, ow), dtype=torch.uint8, device=self.device)

    def flush(self):
        """End of the stream (temporal mode): drains BSVD's pipeline (the reference feeds None, bsvd/model.py:555-569) and
        returns the entries of the jobs still in flight, oldest first; the next frame starts a new clip."""
        if not self._temporal() or self._den_stream is None:
            return []
        with torch.cuda.device(self.device):
            return self._flush()

    def _flush(self):
        for den in self._den_stream.flush():
            self._ready.append(self._finish_single(den, self._lr_fifo.popleft()))
        self._den_stream.reset()
        self.lr_prev = None
        out = []
        while self._jobs:
            out.append(self._pop_delayed())
        return out

    # ------------------------------------------------------------------ glue helpers (csrc/glue.cu)
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _stats(self, img, n, c, h, w, slot):
        key = (slot, n * c)
        buf = self._sums.get(key)
        if buf is None:
            buf = self._sums[key] = torch.empty(n * c, 2, dtype=torch.float64, device=self.device)
        L.check(self.lib.ss4k_glue_chan_stats(_ptr(img), _fmt(img), n, c, h, w, _ptr(buf), self._stream()))
        return buf

    def _area(self, img, n, c, h, w, oh, ow):
        out = torch.empty(n, c, oh, ow, dtype=torch.float32, device=self.device)
        L.check(self.lib.ss4k_glue_area_pool(_ptr(img), _fmt(img), n, c, h, w, _ptr(out), oh, ow, self._stream()))
        return out

    def _finish(self, hr, n, h, w, diff, hs, ls, cnt_hr, cnt_lr, want_resize):
        """The colour-matched frames [n, *frame_shape] in out_fmt.  NV12: the finalising kernels store NV12 themselves
        (fused resize: finalize_bicubic_nv12, no resize: finalize_nv12); the two-pass resize for downscale factors above
        2 (e.g. lr_level 5: 4320p -> 1440p; off the live path) converts its uint8 RGB frame with Engine.rgb_to_nv12."""
        dh, dw = (diff.shape[-2], diff.shape[-1]) if diff is not None else (0, 0)
        st = self._stream()
        nv12 = self.out_fmt == L.FMT_NV12
        oh, ow = self.output_shape if want_resize else (h, w)
        shape = (n,) + frame_shape(self.out_fmt, oh, ow)   # raises before any launch when NV12 cannot hold (oh, ow)
        if want_resize:
            if h <= 2 * oh and w <= 2 * ow:
                out = torch.empty(shape, dtype=torch.uint8, device=self.device)
                # clamp(match - colour diff) and the bicubic resize (:214-231) in one pass over the net's output
                entry = self.lib.ss4k_glue_finalize_bicubic_nv12 if nv12 else self.lib.ss4k_glue_finalize_bicubic_u8
                L.check(entry(_ptr(hr), _fmt(hr), n, 3, h, w, _ptr(diff), dh, dw, _ptr(hs), _ptr(ls), cnt_hr, cnt_lr, _ptr(out),
                              oh, ow, 0, st))
                return out
            tmp = torch.empty(n, 3, h, w, dtype=torch.float32, device=self.device)   # downscale > 2: two passes
            L.check(self.lib.ss4k_glue_finalize(_ptr(hr), _fmt(hr), n, 3, h, w, _ptr(diff), dh, dw, _ptr(hs), _ptr(ls),
                                                cnt_hr, cnt_lr, None, _ptr(tmp), 0, st))
            rgb = torch.empty(n, oh, ow, 3, dtype=torch.uint8, device=self.device)
            L.check(self.lib.ss4k_glue_bicubic_u8(_ptr(tmp), n, 3, h, w, _ptr(rgb), oh, ow, 0, st))
            return self.engine.rgb_to_nv12(rgb).view(shape) if nv12 else rgb
        out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        entry_args = (_ptr(hr), _fmt(hr), n, 3, h, w, _ptr(diff), dh, dw, _ptr(hs), _ptr(ls), cnt_hr, cnt_lr, _ptr(out))
        if nv12:
            L.check(self.lib.ss4k_glue_finalize_nv12(*entry_args, 0, st))
        else:
            L.check(self.lib.ss4k_glue_finalize(*entry_args, None, 0, st))
        return out

    def _run_model(self, lr):
        """model(lr): lr is uint8 NHWC or float NCHW on the device; returns fp16 NCHW."""
        if lr.dtype == torch.uint8:
            n, h, w, _ = lr.shape
            return self.model._plan(n, h, w, L.FMT_U8_NHWC, L.FMT_F16_NCHW).run(lr)
        return self.model(lr)

    # ------------------------------------------------------------------ upscale (fsrcnn_upscaler.py:144-166)
    def upscale(self, frames):
        with torch.cuda.device(self.device):     # the glue kernels launch on the current device's stream
            return self._upscale(frames)

    def _upscale(self, frames):
        assert isinstance(frames, torch.Tensor)
        if frames.device != self.device:
            frames = frames.to(self.device, non_blocking=True)
        if frames.ndim != 4:
            raise Exception(frames.shape)
        assert frames.shape[-1] == 3
        frames = frames.contiguous()
        if self._temporal():
            return self.upscale_temporal(frames)
        if self.single_mode:
            return torch.stack([self.upscale_single(frames[i]) for i in range(frames.shape[0])], dim=0)
        return self.upscale_multi(frames)

    def upscale_temporal(self, frames):
        """upscale_single with BSVD as a temporal stream: pushes the job's frames into the ring-buffer engine and returns
        the frames that left it (none for the first 16 frames, then one per frame; flush() returns the tail)."""
        lh, lw = self.lr_shape
        if self._den_stream is None:
            if self.denoise_model is None:
                self._build_denoiser()
            self._den_stream = self.denoise_model.stream(lh, lw, max_frames=_TEMPORAL_PUSH)
        n, ih, iw, _ = frames.shape
        lr_before = self._area(frames, n, 3, ih, iw, lh, lw)
        x = torch.empty(n, 4, lh, lw, dtype=torch.float32, device=self.device)
        x[:, :3].copy_(lr_before)
        x[:, 3].fill_(0.1 * self.denoise_rate)                                   # :262,269
        if self.lr_prev is None:
            x[0, 3].fill_(0.05)
        self.lr_prev = lr_before[n - 1:n]
        done = []
        for i0 in range(0, n, _TEMPORAL_PUSH):
            i1 = min(n, i0 + _TEMPORAL_PUSH)
            self._lr_fifo.extend(lr_before[i:i + 1] for i in range(i0, i1))
            self.profiler.start('fsrcnn.denoise')
            den = self._den_stream.push_frames(x[i0:i1])
            self.profiler.end('fsrcnn.denoise')
            for j in range(den.shape[0]):
                done.append(self._finish_single(den[j:j + 1], self._lr_fifo.popleft()))
        if done:
            return torch.stack(done, dim=0)
        return self._no_frames()

    def upscale_multi(self, img):
        """fsrcnn_upscaler.py:168-233"""
        n, ih, iw, _ = img.shape
        lh, lw = ih, iw
        lr = img
        if (iw > self.lr_shape[-1] or ih > self.lr_shape[-2]) and self.lr_hr_resize:
            lh, lw = self.lr_shape
            lr = self._area(img, n, 3, ih, iw, lh, lw)                       # :173-176
        self.profiler.start('fsrcnn.model')
        hr = self._run_model(lr)                                             # :181
        self.profiler.end('fsrcnn.model')
        h, w = hr.shape[-2], hr.shape[-1]
        hs = self._stats(hr, n, 3, h, w, 'hr')                               # :188-199
        ls = self._stats(lr, n, 3, lh, lw, 'lr')
        diff = None
        if (h // 8) > (self.match_blur.shape[-1] // 2) and h > 64 and w > 64:   # :203
            hb = self._area(hr, n, 3, h, w, h // 8, w // 8)
            lb = self._area(lr, n, 3, lh, lw, h // 8, w // 8)
            diff = torch.empty_like(hb)
            L.check(self.lib.ss4k_glue_blur_diff(_ptr(hb), _ptr(lb), _ptr(diff), _ptr(self.match_blur), self.match_blur.shape[-1],
                                                 n, 3, h // 8, w // 8, _ptr(hs), _ptr(ls), float(h * w), float(lh * lw),
                                                 self._stream()))
        resize = (self.output_shape is not None) and self.lr_hr_resize and tuple(self.output_shape) != (h, w)
        return self._finish(hr, n, h, w, diff, hs, ls, float(h * w), float(lh * lw), resize)

    def upscale_single(self, img):
        """fsrcnn_upscaler.py:235-326 (one frame, optional BSVD denoise in front of the upscaler)"""
        ih, iw, _ = img.shape
        lh, lw = self.lr_shape
        lr_before = self._area(img.unsqueeze(0), 1, 3, ih, iw, lh, lw)        # :237-241 (always area-resized)
        den = None
        if self.denoising:
            x = torch.empty(1, 1, 4, lh, lw, dtype=torch.float32, device=self.device)
            first = self.lr_prev is None
            x[0, 0, :3].copy_(lr_before[0])
            x[0, 0, 3].fill_(0.05 if first else 0.1 * self.denoise_rate)       # :262,269
            self.profiler.start('fsrcnn.denoise')
            if self.denoise_model is None:
                self._build_denoiser()
            den = self.denoise_model(x)[:, -1]                                 # :277  (F = 1 clip)
            self.profiler.end('fsrcnn.denoise')
            self.lr_prev_diff_map = x[0, 0, 3]
        return self._finish_single(den, lr_before)

    def _finish_single(self, den, lr_before):
        """The rest of upscale_single for one frame: den [1,3,lh,lw] is BSVD's output for it (None: denoising off)."""
        lh, lw = self.lr_shape
        lr = lr_before
        if den is not None:
            lr = torch.empty(1, 3, lh, lw, dtype=torch.float32, device=self.device)
            L.check(self.lib.ss4k_glue_sharpen_blend(_ptr(den), _fmt(den), 1, 3, lh, lw, 0.00002, 0.8, _ptr(lr_before), 0,
                                                     _ptr(lr), self._stream()))   # :278-281
            self.lr_prev = lr
        self.profiler.start('fsrcnn.model')
        hr = self.model(lr)                                                     # :293-295
        h, w = hr.shape[-2], hr.shape[-1]
        if den is not None:
            hs_in = hr
            hr = torch.empty(1, 3, h, w, dtype=torch.float32, device=self.device)
            L.check(self.lib.ss4k_glue_sharpen_blend(_ptr(hs_in), _fmt(hs_in), 1, 3, h, w, 0.00007, 1.0, None, 0, _ptr(hr),
                                                     self._stream()))           # :298-299
        self.profiler.end('fsrcnn.model')
        hs = self._stats(hr, 1, 3, h, w, 'hr1')                                  # :302-313
        ls = self._stats(lr_before, 1, 3, lh, lw, 'lr1')
        resize = (self.output_shape is not None) and tuple(self.output_shape) != (h, w)
        return self._finish(hr, 1, h, w, None, hs, ls, float(h * w), float(lh * lw), resize)[0]
