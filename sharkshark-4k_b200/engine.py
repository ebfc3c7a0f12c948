"""Thin Python host layer over the C ABI: contexts, weight upload, plans.

PyTorch is used only for device buffers and streams; all arithmetic runs in libss4k.so.
"""
import ctypes
import struct
import json

import torch

from . import _lib as L


class Engine:
    """One engine per CUDA device (== one FsrcnnUpscalerService process in the reference,
    src/upscale/fsrcnn_upscaler.py:118-139)."""

    _by_device = {}

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise L.Ss4kError("no CUDA device: the ss4k engine has no CPU fallback")
        self.lib = L.load()
        self.device = torch.device("cuda", int(device) if not isinstance(device, torch.device) else (device.index or 0))
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self.lib.ss4k_create(self.device.index, ctypes.byref(h)))
        self.h = h
        self._next_net = 0

    @classmethod
    def get(cls, device=0):
        idx = device.index if isinstance(device, torch.device) else int(device)
        idx = idx or 0
        if idx not in cls._by_device:
            cls._by_device[idx] = Engine(idx)
        return cls._by_device[idx]

    @property
    def desc_mode(self):
        return self.lib.ss4k_desc_mode(self.h)

    @property
    def launch_count(self):
        return self.lib.ss4k_launch_count(self.h)

    def new_net(self, state_dict):
        """Upload a state dict (OIHW fp32 tensors, reference key names) into a fresh weight slot."""
        net_id = self._next_net
        self._next_net += 1
        for name, t in state_dict.items():
            t = t.detach().to("cpu", torch.float32).contiguous()
            if t.ndim == 0:
                t = t.reshape(1)
            if t.ndim > 4:
                continue
            shape = (ctypes.c_int64 * t.ndim)(*t.shape)
            L.check(self.lib.ss4k_load_weights(self.h, net_id, name.encode(), ctypes.c_void_p(t.data_ptr()),
                                               L.DT_F32, shape, t.ndim), self.h)
        return net_id

    def release_net(self, net_id):
        """Drop the host (fp32) copy of a net's weights; plans already created keep their packed device weights."""
        if self.h:
            self.lib.ss4k_clear_weights(self.h, net_id)

    def plan(self, net_id, arch, n, h, w, scale=4, depth=0, tile=0, tile_pad=10, act_mode=L.ACT_F16,
             in_fmt=L.FMT_F32_NCHW, out_fmt=L.FMT_F32_NCHW, use_graph=True, bsvd_noise=0.0, pre_pad=0, own=None):
        cfg = make_cfg(net_id, arch, n, h, w, scale, depth, tile, tile_pad, act_mode, in_fmt, out_fmt, use_graph)
        cfg.reserved[0] = struct.unpack("<i", struct.pack("<f", float(bsvd_noise)))[0]
        cfg.reserved[1] = int(pre_pad)
        if own is not None:   # BSVD: frames [lo, hi) of the clip are wanted, the rest is temporal halo
            cfg.reserved[2], cfg.reserved[3] = int(own[0]), int(own[1])
        return Plan(self, cfg)

    def rgb_to_nv12(self, frames):
        """uint8 NHWC RGB CUDA frames [N,H,W,3] -> uint8 [N, H*W*3/2] NV12 (Y plane + interleaved UV), BT.709 limited
        range (encoder side of the colour stage; ss4k_rgb_to_nv12)."""
        assert frames.is_cuda and frames.dtype == torch.uint8 and frames.is_contiguous() and frames.shape[-1] == 3
        n, h, w, _ = frames.shape
        out = torch.empty(n, h * w * 3 // 2, device=frames.device, dtype=torch.uint8)
        st = ctypes.c_void_p(torch.cuda.current_stream(frames.device).cuda_stream)
        L.check(self.lib.ss4k_rgb_to_nv12(self.h, ctypes.c_void_p(frames.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                          n, h, w, st), self.h)
        return out

    def _surfaces(self, surfaces):
        arr = (L.Nv12Surface * len(surfaces))()
        for i, (y, uv) in enumerate(surfaces):   # 2-D uint8 CUDA views with unit inner stride: pitch = stride(0)
            assert y.is_cuda and uv.is_cuda and y.dtype == uv.dtype == torch.uint8 and y.stride(1) == 1 and uv.stride(1) == 1
            arr[i].y, arr[i].uv = y.data_ptr(), uv.data_ptr()
            arr[i].pitch_y, arr[i].pitch_uv = y.stride(0), uv.stride(0)
        return arr

    def nv12_pack(self, surfaces, h, w, out=None):
        """Pitched NV12 decoder surfaces [(y_plane, uv_plane), ...] -> the packed chunk [n, h*3/2, w] the plans read
        (ss4k_nv12_pack: 2-D DMA copies, stream-ordered)."""
        n = len(surfaces)
        if out is None:
            out = torch.empty(n, h * 3 // 2, w, dtype=torch.uint8, device=self.device)
        st = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        L.check(self.lib.ss4k_nv12_pack(self.h, self._surfaces(surfaces), n, h, w, ctypes.c_void_p(out.data_ptr()), st), self.h)
        return out

    def nv12_unpack(self, packed, surfaces, h, w):
        """Packed NV12 frames -> pitched encoder input surfaces (ss4k_nv12_unpack)."""
        st = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        L.check(self.lib.ss4k_nv12_unpack(self.h, ctypes.c_void_p(packed.data_ptr()), self._surfaces(surfaces), len(surfaces), h, w, st),
                self.h)

    def conv3x3(self, x, weight, bias=None, slope=None, residual=None, mode=L.MODE_CONV3, act=0,
                act_mode=L.ACT_F16, pixel_shuffle=0, alpha=1.0, beta=1.0, direct_f32=False):
        """Operator-level entry (kernel parity tests): float NCHW CUDA tensors in / out."""
        n, cin, h, w = x.shape
        cout = weight.shape[0]
        oh, ow = h, w
        if mode == L.MODE_UP2:
            oh, ow = 2 * h, 2 * w
        elif mode == L.MODE_S2:
            oh, ow = h // 2, w // 2
        oc = cout
        if pixel_shuffle:
            oc, oh, ow = cout // (pixel_shuffle ** 2), oh * pixel_shuffle, ow * pixel_shuffle
        y = torch.empty(n, oc, oh, ow, device=x.device, dtype=torch.float32)
        d = L.ConvDesc()
        d.struct_size = ctypes.sizeof(L.ConvDesc)
        d.n, d.h, d.w, d.cin, d.cout = n, h, w, cin, cout
        d.mode, d.act, d.act_mode, d.pixel_shuffle = mode, act, act_mode, pixel_shuffle
        d.alpha, d.beta = alpha, beta
        d.reserved[0] = 1 if direct_f32 else 0
        ts = [t.contiguous().float() if t is not None else None for t in (x, weight, bias, slope, residual)]
        ptr = [ctypes.c_void_p(t.data_ptr()) if t is not None else None for t in ts]
        st = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        L.check(self.lib.ss4k_conv3x3(self.h, ctypes.byref(d), ptr[0], ptr[1], ptr[2], ptr[3], ptr[4],
                                      ctypes.c_void_p(y.data_ptr()), st), self.h)
        return y


def make_cfg(net_id, arch, n, h, w, scale=4, depth=0, tile=0, tile_pad=10, act_mode=L.ACT_F16,
             in_fmt=L.FMT_F32_NCHW, out_fmt=L.FMT_F32_NCHW, use_graph=True):
    c = L.PlanCfg()
    c.struct_size = ctypes.sizeof(L.PlanCfg)
    c.net_id, c.arch, c.n, c.h, c.w = net_id, arch, n, h, w
    c.scale, c.depth, c.tile, c.tile_pad = scale, depth, tile, tile_pad
    c.act_mode, c.in_fmt, c.out_fmt, c.use_graph = act_mode, in_fmt, out_fmt, 1 if use_graph else 0
    return c


def plan_dry(cfg):
    """Host-only lowering of a configuration to its layer program (works without a GPU)."""
    lib = L.load()
    out = ctypes.c_void_p()
    L.check(lib.ss4k_plan_dry(ctypes.byref(cfg), ctypes.byref(out)))
    try:
        return json.loads(ctypes.string_at(out).decode())
    finally:
        lib.ss4k_free(out)


def tile_layout(cfg):
    """Host-only: RealESRGANer's tile grid for a configuration (tile, tile_pad, reserved[1] = pre_pad) and its packing into
    crop atlases, as the engine's tiled plan would run it (works without a GPU)."""
    lib = L.load()
    out = ctypes.c_void_p()
    L.check(lib.ss4k_debug_tile_layout(ctypes.byref(cfg), ctypes.byref(out)))
    try:
        return json.loads(ctypes.string_at(out).decode())
    finally:
        lib.ss4k_free(out)


class PlanCache:
    """Shape-keyed LRU cache of engine plans.  A plan owns its workspaces (about 2 GB for RRDBNet at 720p), so a
    caller that sees arbitrary shapes -- the reference's still-image server drives the same service with one plan
    per image size (src/sharkshark/image_server/image_pipeline.py:54-64) -- must not keep every plan alive: the
    least recently used plan is destroyed once `max_plans` are cached."""

    def __init__(self, max_plans=8):
        self.max_plans = max(1, int(max_plans))
        self._d = {}        # insertion order == recency order
        self.evictions = 0

    def get(self, key, make):
        p = self._d.pop(key, None)
        if p is None:
            while len(self._d) >= self.max_plans:
                old = self._d.pop(next(iter(self._d)))
                self.evictions += 1
                close = getattr(old, "close", None)
                if close is not None:
                    close()
            p = make()
        self._d[key] = p
        return p

    def __len__(self):
        return len(self._d)

    def __contains__(self, key):
        return key in self._d


_OUT_DTYPES = {L.FMT_F32_NCHW: torch.float32, L.FMT_F16_NCHW: torch.float16, L.FMT_U8_NHWC: torch.uint8,
               L.FMT_NV12: torch.uint8}


def out_shape_of(out_fmt, n, c, h, w):
    """Shape of a plan's output tensor for ss4k_plan_out_shape's (n, c, h, w): NHWC for uint8 RGB, packed NV12 frames
    [n, h*3/2, w] (Y plane, then interleaved UV) for NV12, NCHW otherwise."""
    if out_fmt == L.FMT_U8_NHWC:
        return (n, h, w, c)
    if out_fmt == L.FMT_NV12:
        return (n, h * 3 // 2, w)
    return (n, c, h, w)


class Plan:
    def __init__(self, engine, cfg):
        self.engine, self.cfg = engine, cfg
        self.lib = engine.lib
        h = ctypes.c_void_p()
        with torch.cuda.device(engine.device):
            L.check(self.lib.ss4k_plan_create(engine.h, ctypes.byref(cfg), ctypes.byref(h)), engine.h)
        self.h = h
        shp = (ctypes.c_int32 * 4)()
        self.lib.ss4k_plan_out_shape(h, ctypes.byref(shp))
        self.out_nchw = tuple(shp)
        self.flops = self.lib.ss4k_plan_flops(h)
        self.launches = self.lib.ss4k_plan_launches(h)
        self.graph_steps = self.lib.ss4k_plan_graph_steps(h)
        self.steps = self.lib.ss4k_plan_steps(h)
        ib, ob = ctypes.c_int64(), ctypes.c_int64()
        self.lib.ss4k_plan_io_bytes(h, ctypes.byref(ib), ctypes.byref(ob))
        self.in_bytes, self.out_bytes = ib.value, ob.value

    def out_shape(self):
        return out_shape_of(self.cfg.out_fmt, *self.out_nchw)

    def new_output(self):
        return torch.empty(self.out_shape(), device=self.engine.device, dtype=_OUT_DTYPES[self.cfg.out_fmt])

    def run(self, x, out=None):
        """x: CUDA tensor in the plan's in_fmt layout; returns a CUDA tensor (stream-ordered, no sync)."""
        assert x.is_cuda and x.is_contiguous()
        assert x.numel() * x.element_size() == self.in_bytes, (x.shape, x.dtype, self.in_bytes)
        if out is None:
            out = self.new_output()
        st = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        L.check(self.lib.ss4k_run(self.h, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(out.data_ptr()), st),
                self.engine.h)
        return out

    def input_act(self):
        """(device pointer, channel pitch, pixel-unshuffle factor, is_bf16) of the tensor the plan's layout step writes
        (ss4k_plan_input_act); raises for plans without a plain layout step."""
        ptr, pitch, us, bf = ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        L.check(self.lib.ss4k_plan_input_act(self.h, ctypes.byref(ptr), ctypes.byref(pitch), ctypes.byref(us), ctypes.byref(bf)),
                self.engine.h)
        return ptr.value, pitch.value, us.value, bf.value

    def run_act(self, out):
        """The plan without its layout step: the caller has written the first-layer activation tensor (input_act())."""
        st = ctypes.c_void_p(torch.cuda.current_stream(out.device).cuda_stream)
        L.check(self.lib.ss4k_run_act(self.h, ctypes.c_void_p(out.data_ptr()), st), self.engine.h)
        return out

    def profile(self, x, out=None):
        """One un-graphed run with a CUDA event between every step: list of (ms, flops, kind) per step
        (kind 0 layout/colour kernel, 1 row-streaming conv kernel, 2 tile conv kernel, 4 a layout step done by the
        first conv's loader: no launch of its own).  An NV12-output plan whose last conv does not store NV12 itself ends with the uint8 RGB -> NV12 conversion (kind 0)."""
        if out is None:
            out = self.new_output()
        cap = self.steps + 8
        ms, fl, kd = (ctypes.c_float * cap)(), (ctypes.c_double * cap)(), (ctypes.c_int32 * cap)()
        st = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        n = self.lib.ss4k_plan_profile(self.h, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(out.data_ptr()), st,
                                       ms, fl, kd, cap)
        if n < 0:
            L.check(n, self.engine.h)
        return [(ms[i], fl[i], kd[i]) for i in range(n)]

    def run_host(self, x_host, out_host):
        """Host (pinned) tensors in / out: H2D + run + D2H inside the call (bench.py e2e)."""
        assert not x_host.is_cuda and not out_host.is_cuda
        L.check(self.lib.ss4k_run_host(self.h, ctypes.c_void_p(x_host.data_ptr()),
                                       ctypes.c_void_p(out_host.data_ptr())), self.engine.h)
        return out_host

    def run_host_async(self, x_host, out_host):
        """Pipelined form of run_host: queues H2D + run + D2H and returns; successive calls overlap their copies with
        each other's kernels.  Alternate between two pinned `out_host` buffers and call host_sync() before reading."""
        assert not x_host.is_cuda and not out_host.is_cuda
        L.check(self.lib.ss4k_run_host_async(self.h, ctypes.c_void_p(x_host.data_ptr()),
                                             ctypes.c_void_p(out_host.data_ptr())), self.engine.h)

    def host_sync(self):
        L.check(self.lib.ss4k_plan_host_sync(self.h), self.engine.h)

    def close(self):
        if self.h:
            self.lib.ss4k_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
