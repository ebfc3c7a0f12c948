"""Drop-in for the reference's BSVD denoiser factory
(reference: src/upscale/model/bsvd/factory.py:21-83 build_model; src/upscale/model/bsvd/model.py:467-588 BSVD).

``build_model(device, input_shape, jit_mode)`` keeps the reference signature and returns an ``nn.Module`` whose
``forward(x)`` takes ``[N, F, 4, H, W]`` (noisy RGB + noise map, as fsrcnn_upscaler.py:262-277 builds it) and returns
``[N, F, 3, H, W]``.  Like the reference (model.py:519-520) the N*F frames are ONE stream; each call is a
self-contained clip (pipeline filled, drained and reset, model.py:555-580).  All arithmetic runs in libss4k.so.
"""
import os

import torch
from torch import nn

from . import _lib as L
from .engine import Engine, PlanCache


def load_checkpoint(path):
    """BSVD.load (model.py:487-499): ckpt['params'], prefix [module.]base_model.nets_list.{0,1}. -> temp1. / temp2.;
    DownBlock / UpBlock / MemCvBlock key renames of model.py:167-169,276-279,304-306."""
    ck = torch.load(path, map_location="cpu")["params"]
    base = "module.base_model." if "module" in next(iter(ck)) else "base_model."
    out = {}
    for k, v in ck.items():
        for i, t in ((0, "temp1."), (1, "temp2.")):
            pre = f"{base}nets_list.{i}."
            if not k.startswith(pre):
                continue
            r = k[len(pre):]
            blk, rest = r.split(".", 1)
            if blk in ("downc0", "downc1"):
                if rest.startswith("convblock.0."):
                    rest = rest
                elif rest.startswith("convblock.3."):
                    rest = "memconv." + rest[len("convblock.3."):].replace("net.", "op.conv.")
                else:
                    continue
            elif blk in ("upc2", "upc1"):
                if rest.startswith("convblock.1."):
                    rest = "convblock.0." + rest[len("convblock.1."):]
                elif rest.startswith("convblock.0."):
                    rest = "memconv." + rest[len("convblock.0."):].replace("net.", "op.conv.")
                else:
                    continue
            out[t + blk + "." + rest] = v
    return out


def pick_act_mode(state_dict):
    """fp16 single-MMA operands pass the parity gate for trained-like weight magnitudes; weights with the gain of
    the reference constructor's ``kaiming_normal_`` init (model.py:393-400,501-508: fan_in * var(W) == 2, outputs
    span +-14 in fp32) need the hi/lo split mode (SURVEY.md section 7 H2).  Decision: median over the 3x3 convs of
    fan_in * var(W) above 1.2 -> split."""
    gains = []
    for k, v in state_dict.items():
        if k.endswith(".weight") and v.dim() == 4:
            fan_in = v.shape[1] * v.shape[2] * v.shape[3]
            gains.append(float(v.float().var().item()) * fan_in)
    if not gains:
        return L.ACT_F16
    gains.sort()
    return L.ACT_F16_SPLIT if gains[len(gains) // 2] > 1.2 else L.ACT_F16


class NativeBSVD(nn.Module):
    """BSVD(chns=[32,64,128], mid_ch=32, interm_ch=30, act='relu6', norm='none') on the native engine."""

    shift_num = 16  # BSVD.count_shift (model.py:582-588): 16 BiBufferConvs -> +-16 frame receptive field

    def __init__(self, state_dict, device=0, act_mode=L.ACT_F16, out_dtype=torch.float32, use_graph=True, max_plans=12):
        super().__init__()
        self.engine = Engine.get(device)
        if act_mode == "auto":
            act_mode = pick_act_mode(state_dict)
        self.act_mode, self.out_dtype, self.use_graph = act_mode, out_dtype, use_graph
        self.net_id = self.engine.new_net(state_dict)
        self._plans = PlanCache(max_plans)

    def _plan(self, t, h, w, in_fmt, out_fmt, noise=0.0, own=None):
        """own = (lo, hi): only frames [lo, hi) of the t-frame clip are wanted (the others are the temporal halo of a
        sharded stream, sharding.bsvd_chunks): every layer then runs only on the frames the owned outputs depend on
        (csrc/bsvd_program.cpp) and the plan returns hi - lo frames."""
        if own is not None and tuple(own) == (0, t):
            own = None
        key = (t, h, w, in_fmt, out_fmt, float(noise), tuple(own) if own is not None else None)
        return self._plans.get(key, lambda: self.engine.plan(
            self.net_id, L.ARCH_BSVD, t, h, w, act_mode=self.act_mode, in_fmt=in_fmt, out_fmt=out_fmt,
            use_graph=self.use_graph, bsvd_noise=noise, own=own))

    def denoise_frames(self, frames, h, w, noise, nv12=False, own=None):
        """Frame-format entry: a clip of uint8 NHWC RGB frames ``[T,h,w,3]`` or NV12 frames ``[T, h*w*3/2]`` (CUDA) ->
        ``[T,3,h,w]`` (``[hi-lo,3,h,w]`` with ``own=(lo, hi)``); /255, NV12 -> RGB and the constant noise map
        (0.1 * denoise_rate, fsrcnn_upscaler.py:262) are produced by the engine's layout kernel."""
        t = frames.shape[0]
        out_fmt = L.FMT_F16_NCHW if self.out_dtype == torch.float16 else L.FMT_F32_NCHW
        return self._plan(t, h, w, L.FMT_NV12 if nv12 else L.FMT_U8_NHWC, out_fmt, noise, own=own).run(frames.contiguous())

    def forward(self, x, noise_map=None):
        if noise_map is not None:
            x = torch.cat([x, noise_map], dim=2)
        if not x.is_cuda:
            raise L.Ss4kError("native BSVD called with a CPU tensor: there is no CPU path")
        n, f, c, h, w = x.shape
        if c != 4:
            raise ValueError("BSVD input is [N, F, 4, H, W] (RGB + noise map)")
        if x.dtype not in (torch.float16, torch.float32):
            x = x.float()
        x = x.reshape(n * f, c, h, w).contiguous()
        in_fmt = L.FMT_F16_NCHW if x.dtype == torch.float16 else L.FMT_F32_NCHW
        out_fmt = L.FMT_F16_NCHW if self.out_dtype == torch.float16 else L.FMT_F32_NCHW
        out = self._plan(n * f, h, w, in_fmt, out_fmt).run(x)
        return out.reshape(n, f, 3, h, w)

    def stream(self, h, w, in_fmt=L.FMT_F32_NCHW, noise=0.0, max_frames=1):
        """A frame-at-a-time stream in this model's precision mode (the split precision mode included).  ``in_fmt``:
        ``FMT_F32_NCHW`` frames ``[4,h,w]`` (RGB + noise map, the reference layout) or ``FMT_U8_NHWC`` / ``FMT_NV12``
        frames with the constant noise map ``noise`` filled in by the layout kernel.  ``max_frames``: the most frames one
        ``push_frames`` call may carry (every ring then holds ``max_frames - 1`` more frames)."""
        return BSVDStream(self, h, w, in_fmt, noise, max_frames)

    def streaming_forward(self, input_seq):
        """BSVD.streaming_forward (model.py:526-580) through the ring-buffer engine: feed, drain, reset."""
        if isinstance(input_seq, torch.Tensor):
            input_seq = [input_seq[i:i + 1] for i in range(input_seq.shape[0])]
        _, _, h, w = input_seq[0].shape
        s = self.stream(h, w)
        outs = [o for o in (s.push(x) for x in input_seq) if o is not None]
        outs += list(s.flush())
        s.close()
        return torch.cat(outs, dim=0)

    def close(self):
        """Destroy the cached plans and release the engine's host copy of the weights (ss4k_clear_weights)."""
        for p in list(self._plans._d.values()):
            p.close()
        self._plans._d.clear()
        if self.net_id is not None:
            self.engine.release_net(self.net_id)
            self.net_id = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        """Every forward() is a complete clip, so there is no state to reset (model.py:482-484,579)."""

    def half(self):
        return self

    def float(self):
        return self


class BSVDStream:
    """Frame-at-a-time denoising with persistent ring buffers in HBM (BSVD.feedin_one_element, model.py:510-513):
    ``push(frame)`` returns the denoised frame t-16 once the 16-stage pipeline is full, else None; ``flush()``
    yields the remaining frames (the reference feeds ``None``, model.py:555-569); ``reset()`` starts a new clip.
    ``push_frames(frames)`` pushes up to ``max_frames`` consecutive frames in one call (each conv runs once over them)."""

    def __init__(self, model, h, w, in_fmt=L.FMT_F32_NCHW, noise=0.0, max_frames=1):
        import ctypes
        self.model, self.h, self.w, self.in_fmt, self.max_frames = model, h, w, in_fmt, max_frames
        self.lib = model.engine.lib
        self.plan = model._plan(1, h, w, in_fmt, L.FMT_F32_NCHW, noise)
        hdl = ctypes.c_void_p()
        L.check(self.lib.ss4k_bsvd_stream_open_batched(self.plan.h, max_frames, ctypes.byref(hdl)), model.engine.h)
        self.hdl = hdl
        self.latency = self.lib.ss4k_bsvd_stream_latency(hdl)

    def _st(self, dev):
        import ctypes
        return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def push(self, frame):
        import ctypes
        if self.in_fmt == L.FMT_F32_NCHW:
            x = frame.reshape(4, self.h, self.w).float().contiguous()
        else:  # uint8 RGB [h,w,3] or NV12 [h*3/2, w]: decoded, normalised and extended by the noise map on the device
            if frame.dtype != torch.uint8:
                raise ValueError("frame-format streams take uint8 frames")
            x = frame.contiguous()
        out = torch.empty(1, 3, self.h, self.w, device=x.device, dtype=torch.float32)
        got = ctypes.c_int(0)
        L.check(self.lib.ss4k_bsvd_stream_push(self.hdl, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                               ctypes.byref(got), self._st(x.device)), self.model.engine.h)
        return out if got.value else None

    def push_frames(self, frames):
        """Frames t .. t+n-1 of the stream: ``[n,4,h,w]`` float, ``[n,h,w,3]`` uint8 RGB or ``[n,h*3/2,w]`` NV12, with
        1 <= n <= max_frames.  Returns the denoised frames that fell out, oldest first: ``[m,3,h,w]`` float, m may be 0."""
        import ctypes
        n = frames.shape[0]
        if self.in_fmt == L.FMT_F32_NCHW:
            x = frames.reshape(n, 4, self.h, self.w).float().contiguous()
        else:
            if frames.dtype != torch.uint8:
                raise ValueError("frame-format streams take uint8 frames")
            x = frames.contiguous()
        out = torch.empty(n, 3, self.h, self.w, device=x.device, dtype=torch.float32)
        got = ctypes.c_int(0)
        L.check(self.lib.ss4k_bsvd_stream_push_frames(self.hdl, ctypes.c_void_p(x.data_ptr()), n, ctypes.c_void_p(out.data_ptr()),
                                                      ctypes.byref(got), self._st(x.device)), self.model.engine.h)
        return out[:got.value]

    def flush(self):
        import ctypes
        dev = self.model.engine.device
        while True:
            out = torch.empty(1, 3, self.h, self.w, device=dev, dtype=torch.float32)
            got = ctypes.c_int(0)
            L.check(self.lib.ss4k_bsvd_stream_flush(self.hdl, ctypes.c_void_p(out.data_ptr()), ctypes.byref(got), self._st(dev)),
                    self.model.engine.h)
            if not got.value:
                return
            yield out

    def reset(self):
        self.lib.ss4k_bsvd_stream_reset(self.hdl)

    def close(self):
        if self.hdl:
            self.lib.ss4k_bsvd_stream_close(self.hdl)
            self.hdl = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def build_model(device=0, input_shape=(360, 640), jit_mode='ds', state_dict=None, pretrain_ckpt=None,
                act_mode="auto"):
    """Same signature as the reference (bsvd/factory.py:21); ``jit_mode`` is accepted and ignored (every mode
    maps to the native engine).  Weights: ``state_dict`` (reference key names) or a ``bsvd-32.pth`` checkpoint."""
    if state_dict is None:
        path = pretrain_ckpt or './upscale/model/bsvd/bsvd-32.pth'
        if not os.path.isfile(path):
            raise FileNotFoundError(f"{path}: bsvd-32.pth is not shipped with the reference (.MISSING_LARGE_BLOBS); "
                                    "pass state_dict=")
        state_dict = load_checkpoint(path)
    return NativeBSVD(state_dict, device=device, act_mode=act_mode).eval()
