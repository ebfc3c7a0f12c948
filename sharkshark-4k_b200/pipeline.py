"""Denoise + upscale of a frame chunk: the hot path of the reference's live-stream configuration in one call.

Reference composition: src/upscale/fsrcnn_upscaler.py:245-300 (``upscale_single``: BSVD denoiser in front of the
RealESRGAN upscaler, one decoded frame at a time); BASELINE.json configs[2] runs it on an NV12 stream with the
denoiser seeing the frames as ONE temporal stream (BSVD.forward over the chunk, src/upscale/model/bsvd/model.py:515-524)
and the chunks sharded across GPUs with the 16-frame temporal halo (``sharding.bsvd_chunks``).

    NV12 / uint8 RGB frames [T, ...]  --BSVD clip (T frames)-->  half NCHW [T,3,H,W]
        --owned frames: 0.8 * clamp(sharpen(denoised), 0, 1) + 0.2 * decoded frame   (fsrcnn_upscaler.py:278-281)
        -->  RRDBNet / SRVGG, one frame per engine run  -->  uint8 NHWC [n_own, sH, sW, 3]
                                                             or NV12 [n_own, sH*3/2, sW] (RRDBNet, out_fmt=FMT_NV12)

Both nets are engine plans (CUDA graphs of tcgen05 convs) behind the C ABI; colour decode, /255 and the noise map
(0.1 * denoise_rate, fsrcnn_upscaler.py:262) are produced by the BSVD plan's layout kernel, the sharpen / clamp / blend
between the nets by the service glue kernel (csrc/glue.cu, which decodes the NV12 frame for the blend itself).  torch
supplies device buffers, streams and pinned host memory only.

With ``out_fmt=FMT_NV12`` (RRDBNet upscalers) the frames leave as packed NV12 -- the Y plane then interleaved UV, the
layout ``Engine.nv12_unpack`` hands to an encoder's surfaces -- converted by the upscaler's last convolution itself:
bit-identical to the uint8 RGB result followed by ``Engine.rgb_to_nv12``, at half the bytes per frame.
"""
import ctypes

import torch

from . import _lib as L


class DenoiseUpscalePipeline:
    def __init__(self, denoiser, upscaler, h, w, noise, nv12=True, out_fmt=L.FMT_U8_NHWC):
        self.den, self.sr = denoiser, upscaler
        self.h, self.w, self.noise, self.nv12 = h, w, float(noise), nv12
        self.out_fmt = out_fmt
        self.device = denoiser.engine.device
        self.sr_plan = upscaler._plan(1, h, w, L.FMT_F32_NCHW, out_fmt)
        self.lib = denoiser.engine.lib
        # the glue between the nets writes the upscaler's first-layer activation tensor itself (no float image, no layout
        # kernel in the upscaler's plan) unless the plan has no plain layout step (tiled plans)
        try:
            self._act = self.sr_plan.input_act()
        except L.Ss4kError:
            self._act = None
        self._lr = {}
        self._den_out_dtype = denoiser.out_dtype
        self._copy_stream = None
        self._slots = {}
        self._calls = 0

    # ------------------------------------------------------------------ plans
    def den_plan(self, t, lo=0, hi=None):
        """BSVD plan for a t-frame chunk of which frames [lo, hi) are owned (the rest is temporal halo: each layer runs
        only on the frames the owned outputs depend on); returns the owned frames."""
        in_fmt = L.FMT_NV12 if self.nv12 else L.FMT_U8_NHWC
        return self.den._plan(t, self.h, self.w, in_fmt, L.FMT_F16_NCHW, self.noise, own=(lo, t if hi is None else hi))

    def frame_bytes_in(self):
        return self.h * self.w * 3 // 2 if self.nv12 else self.h * self.w * 3

    def out_frame_shape(self):
        return tuple(self.sr_plan.out_shape()[1:])

    def new_output(self, n_own):
        dt = {L.FMT_U8_NHWC: torch.uint8, L.FMT_NV12: torch.uint8, L.FMT_F16_NCHW: torch.float16,
              L.FMT_F32_NCHW: torch.float32}[self.out_fmt]
        return torch.empty((n_own,) + self.out_frame_shape(), device=self.device, dtype=dt)


    # ------------------------------------------------------------------ device-resident path
    def run(self, frames, own=None, out=None, after_frame=None):
        """frames: CUDA uint8 chunk [T, h*w*3/2] (NV12) or [T,h,w,3]; own: slice of the chunk whose frames are
        upscaled (default: all); returns the upscaled frames in the pipeline's out_fmt: [n_own, sH, sW, 3] uint8 RGB,
        [n_own, sH*3/2, sW] uint8 NV12, or [n_own, 3, sH, sW] float / half (stream-ordered, no sync)."""
        with torch.cuda.device(self.device):     # the glue kernel launches on the current device's stream
            return self._run(frames, own, out, after_frame)

    def _run(self, frames, own, out, after_frame):
        t = frames.shape[0]
        own = own if own is not None else slice(0, t)
        lo, hi, _ = own.indices(t)
        frames = frames.contiguous()
        den = self.den_plan(t, lo, hi).run(frames)                # [n_own,3,H,W] half: the owned frames
        if out is None:
            out = self.new_output(hi - lo)
        n_own = hi - lo
        # denoised -> 3x3 reflect sharpen(2e-5) + clamp -> 0.8 * . + 0.2 * original frame (fsrcnn_upscaler.py:278-281)
        st = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        src = frames[lo:hi]
        if self._act is not None:
            ptr, pitch, us, bf = self._act
            den_frame = den.stride(0) * den.element_size()
            src_frame = src.stride(0) * src.element_size()
            for i in range(n_own):
                L.check(self.lib.ss4k_glue_sharpen_blend_act(
                    ctypes.c_void_p(den.data_ptr() + i * den_frame), 1, 1, 3, self.h, self.w, 0.00002, 0.8,
                    ctypes.c_void_p(src.data_ptr() + i * src_frame), 3 if self.nv12 else 2,
                    ctypes.c_void_p(ptr), us, pitch, bf, st), self.den.engine.h)
                self.sr_plan.run_act(out[i:i + 1])
                if after_frame is not None:
                    after_frame(i)
            return out
        lr = self._lr.get(n_own)
        if lr is None:
            lr = self._lr[n_own] = torch.empty(n_own, 3, self.h, self.w, dtype=torch.float32, device=self.device)
        L.check(self.lib.ss4k_glue_sharpen_blend(ctypes.c_void_p(den.data_ptr()), 1, n_own, 3, self.h, self.w,
                                                 0.00002, 0.8, ctypes.c_void_p(src.data_ptr()), 3 if self.nv12 else 2,
                                                 ctypes.c_void_p(lr.data_ptr()), st), self.den.engine.h)
        for i in range(n_own):
            self.sr_plan.run(lr[i:i + 1], out[i:i + 1])
            if after_frame is not None:
                after_frame(i)
        return out

    # ------------------------------------------------------------------ host path (pinned buffers in / out)
    def run_host(self, frames_host, own, out_host):
        """Pinned host chunk in, pinned host frames out (``out_host`` shaped like ``new_output``, any out_fmt).  The H2D copy, both nets and the D2H copies are queued and the
        call returns; the D2H copy of frame i overlaps the upscaling of frame i+1 (copy stream) and consecutive
        calls alternate between two device staging slots.  Call ``host_sync()`` before reading ``out_host``."""
        assert not frames_host.is_cuda and not out_host.is_cuda
        t = frames_host.shape[0]
        lo, hi, _ = own.indices(t)
        key = (t, hi - lo)
        if key not in self._slots:
            self._slots[key] = [{"in": torch.empty(frames_host.shape, dtype=torch.uint8, device=self.device),
                                 "out": self.new_output(hi - lo), "copied": None} for _ in range(2)]
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        slot = self._slots[key][self._calls & 1]
        self._calls += 1
        cur = torch.cuda.current_stream(self.device)
        if slot["copied"] is not None:
            cur.wait_event(slot["copied"])                        # the slot's previous result has left the device
        slot["in"].copy_(frames_host, non_blocking=True)

        def after(i):
            ev = torch.cuda.Event()
            ev.record(cur)
            self._copy_stream.wait_event(ev)
            with torch.cuda.stream(self._copy_stream):
                out_host[i].copy_(slot["out"][i], non_blocking=True)

        self.run(slot["in"], own, slot["out"], after_frame=after)
        done = torch.cuda.Event()
        done.record(self._copy_stream)
        slot["copied"] = done
        return out_host

    def host_sync(self):
        torch.cuda.current_stream(self.device).synchronize()
        if self._copy_stream is not None:
            self._copy_stream.synchronize()
