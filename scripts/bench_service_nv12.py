#!/usr/bin/env python
"""NV12 output of the upscaler service, measured against uint8 RGB output followed by the separate conversion.

The reference's live default: SRVGGNetCompact-32 x4 (seeded random weights), batch 4, 720p frames in, output_shape
(1440, 2560), so the service ends in the fused finalise + bicubic kernel (2880p -> 1440p).  Reports
  * kernel: device time (CUDA events, mean over --iters launches, median over --repeats alternations) of
    (a) ss4k_glue_finalize_bicubic_u8 + ss4k_rgb_to_nv12 and (b) ss4k_glue_finalize_bicubic_nv12, on the arguments the
    service passes for one batch; the two parts of (a) are also timed alone.  The net's fp16 output of one batch is
    354 MB, larger than the 126 MB L2, so every launch reads it from HBM;
  * service: whole-batch upscale() time with uint8 RGB output + Engine.rgb_to_nv12 against the service constructed with
    out_fmt=FMT_NV12 (CUDA events around the call, modes alternated);
  * bytes per output frame, and whether both forms give the same NV12 bytes.
One JSON line on stdout; --out FILE writes it there too.  Needs a B200.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(fns, iters, repeats):
    """{name: median over `repeats` of the mean ms per call over `iters` calls}, the modes alternated."""
    for fn in fns.values():
        event_ms(fn, 2)
    runs = {k: [] for k in fns}
    names = list(fns)
    for r in range(repeats):
        for k in (names if r % 2 == 0 else names[::-1]):
            runs[k].append(event_ms(fns[k], iters))
    return {k: statistics.median(v) for k, v in runs.items()}, runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20, help="launches / batches per timed window")
    ap.add_argument("--repeats", type=int, default=6, help="alternations of the two forms")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_service_nv12.py needs a CUDA device")
    from ss4k_b200 import _lib as L
    from ss4k_b200 import service
    from oracle import srvgg

    torch.manual_seed(0)
    sd = srvgg.SRVGGNetCompact(3, 3, 64, 32, 4).eval().state_dict()
    svcs = {}
    for name, fmt in (("rgb", L.FMT_U8_NHWC), ("nv12", L.FMT_NV12)):
        svc = service.FsrcnnUpscalerService(lr_level=3, device=0, denoising=False, model_name='realesr-general-x4v3',
                                            state_dict=sd, batch_size=4, out_fmt=fmt)
        svc.proc_init()
        svc.output_shape = (1440, 2560)
        svcs[name] = svc
    eng = svcs["rgb"].engine
    n, oh, ow = 4, 1440, 2560
    frames = torch.randint(0, 256, (n, 720, 1280, 3), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(1))

    # ---- the arguments the service hands to its finalising kernel for this batch
    captured = {}
    finish = svcs["rgb"]._finish

    def capture(*a):
        captured["args"] = a
        return finish(*a)
    svcs["rgb"]._finish = capture
    svcs["rgb"].upscale(frames)
    svcs["rgb"]._finish = finish
    hr, n_, h, w, diff, hs, ls, cnt_hr, cnt_lr, _ = captured["args"]
    assert n_ == n and (h, w) == (2880, 5120) and diff is not None
    p = service._ptr
    kargs = (p(hr), service._fmt(hr), n, 3, h, w, p(diff), diff.shape[-2], diff.shape[-1], p(hs), p(ls), cnt_hr, cnt_lr)
    rgb = torch.empty(n, oh, ow, 3, dtype=torch.uint8, device="cuda")
    nv_a = torch.empty(n, oh * 3 // 2, ow, dtype=torch.uint8, device="cuda")
    nv_b = torch.empty_like(nv_a)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fb_u8():
        L.check(eng.lib.ss4k_glue_finalize_bicubic_u8(*kargs, p(rgb), oh, ow, 0, st))

    def to_nv12():
        L.check(eng.lib.ss4k_rgb_to_nv12(eng.h, p(rgb), p(nv_a), n, oh, ow, st), eng.h)

    def form_a():
        fb_u8()
        to_nv12()

    def form_b():
        L.check(eng.lib.ss4k_glue_finalize_bicubic_nv12(*kargs, p(nv_b), oh, ow, 0, st))

    form_a()
    form_b()
    torch.cuda.synchronize()
    kernel_identical = bool(torch.equal(nv_a, nv_b))
    kmed, kruns = alternate({"a": form_a, "b": form_b}, args.iters, args.repeats)
    parts, _ = alternate({"finalize_bicubic_u8": fb_u8, "rgb_to_nv12": to_nv12}, args.iters, args.repeats)

    # ---- whole batch through the service
    def svc_a():
        return eng.rgb_to_nv12(svcs["rgb"].upscale(frames))

    def svc_b():
        return svcs["nv12"].upscale(frames)

    service_identical = bool(torch.equal(svc_a().view(n, oh * 3 // 2, ow), svc_b()))
    smed, sruns = alternate({"a": svc_a, "b": svc_b}, max(1, args.iters // 4), args.repeats)

    line = {
        "metric": "service NV12 output, live default (SRVGG-32 x4, batch 4, 720p -> 2880p -> 1440p): (a) uint8 RGB + "
                  "ss4k_rgb_to_nv12 vs (b) out_fmt NV12",
        "card": card(), "batch": n, "out_frame": f"{ow}x{oh}", "iters": args.iters, "repeats": args.repeats,
        "kernel_us_per_batch": {"a_finalize_bicubic_u8_plus_rgb_to_nv12": 1000 * kmed["a"], "b_finalize_bicubic_nv12": 1000 * kmed["b"],
                                "a_part_finalize_bicubic_u8": 1000 * parts["finalize_bicubic_u8"],
                                "a_part_rgb_to_nv12": 1000 * parts["rgb_to_nv12"],
                                "b_over_a": kmed["b"] / kmed["a"],
                                "runs_a": [1000 * x for x in kruns["a"]], "runs_b": [1000 * x for x in kruns["b"]]},
        "service_ms_per_batch": {"a_rgb_then_rgb_to_nv12": smed["a"], "b_out_fmt_nv12": smed["b"], "b_over_a": smed["b"] / smed["a"],
                                 "runs_a": sruns["a"], "runs_b": sruns["b"]},
        "bytes_per_frame": {"uint8_rgb": oh * ow * 3, "nv12": oh * ow * 3 // 2},
        "nv12_identical": {"kernels": kernel_identical, "service": service_identical},
    }
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
