#!/usr/bin/env python
"""NV12 output of the headline chain, measured against the two-step form it replaces.

cfg3 of bench.py (synthetic NV12 1280x720 chunk -> BSVD-32 split precision -> sharpen / blend glue -> RRDBNet-23 x2),
with the upscaled frames leaving as NV12 for an encoder, in two modes alternated in one process:
  (a) out_fmt uint8 RGB, then ss4k_rgb_to_nv12 on the device (the form the engine offered before NV12 output);
  (b) out_fmt NV12: RRDBNet's last convolution writes NV12 itself.
Reports for each mode: device-resident frames/s (frames and results in HBM), host-path frames/s (pinned NV12 chunk in ->
pinned NV12 frames out, copies inside the timed region), conv_last's launch time from ss4k_plan_profile (+ the separate
conversion kernel in mode a), and the output bytes per frame.  Both modes' NV12 frames are compared byte for byte.
--gpus 2 also times the NCCL gather of one step's finished frames to rank 0 + rank 0's device-to-host copy, for uint8
RGB frames (what mode a moves when it converts after the gather, as bench.py's multi-GPU line does) and for NV12 frames.
One JSON line on stdout; --out FILE writes it there too.  Needs a B200.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402  (cfg3's seeded weights, synthetic stream and constants)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def rgb_to_nv12_into(eng, rgb, nv):
    """ss4k_rgb_to_nv12 of uint8 RGB frames [n, H, W, 3] straight into `nv` (n packed NV12 frames), current stream."""
    import ctypes
    from ss4k_b200 import _lib as L
    n, h, w, _ = rgb.shape
    st = ctypes.c_void_p(torch.cuda.current_stream(rgb.device).cuda_stream)
    L.check(eng.lib.ss4k_rgb_to_nv12(eng.h, ctypes.c_void_p(rgb.data_ptr()), ctypes.c_void_p(nv.data_ptr()), n, h, w, st), eng.h)


def host_step_factory(pipe, eng, frames_host, own, outs_host, convert):
    """pipe.run_host's software pipeline (two device slots, D2H of frame i on a copy stream overlapping frame i+1), with
    the uint8 RGB -> NV12 conversion in front of each frame's copy when `convert` (mode a)."""
    dev = pipe.device
    lo, hi, _ = own.indices(frames_host.shape[0])
    n = hi - lo
    slots = [{"in": torch.empty(frames_host.shape, dtype=torch.uint8, device=dev), "out": pipe.new_output(n),
              "nv": torch.empty((n,) + outs_host[0].shape[1:], dtype=torch.uint8, device=dev), "copied": None} for _ in range(2)]
    cs = torch.cuda.Stream(dev)

    def step(i):
        slot = slots[i & 1]
        out_host = outs_host[i & 1]
        cur = torch.cuda.current_stream(dev)
        if slot["copied"] is not None:
            cur.wait_event(slot["copied"])
        slot["in"].copy_(frames_host, non_blocking=True)

        def after(j):
            src = slot["out"][j]
            if convert:
                rgb_to_nv12_into(eng, slot["out"][j:j + 1], slot["nv"][j:j + 1])
                src = slot["nv"][j]
            ev = torch.cuda.Event()
            ev.record(cur)
            cs.wait_event(ev)
            with torch.cuda.stream(cs):
                out_host[j].copy_(src, non_blocking=True)

        pipe.run(slot["in"], own, slot["out"], after_frame=after)
        done = torch.cuda.Event()
        done.record(cs)
        slot["copied"] = done

    def sync():
        torch.cuda.synchronize()
    return step, sync


def single_gpu(args):
    from ss4k_b200 import _lib as L
    from ss4k_b200 import bsvd as nb, realesrgan, sharding
    from ss4k_b200.pipeline import DenoiseUpscalePipeline

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    F = args.clip
    ch = sharding.bsvd_chunks(F, 1)[0]
    H, W = bench.FRAME_H, bench.FRAME_W
    sr = realesrgan.NativeRRDBNet(bench.oracle_rrdb().state_dict(), scale=bench.SCALE, num_block=bench.BLOCKS, device=0)
    den = nb.NativeBSVD(bench.bsvd_state(1.0), device=0, act_mode=L.ACT_F16_SPLIT, out_dtype=torch.float16)
    eng = sr.engine
    pipes = {"a": DenoiseUpscalePipeline(den, sr, H, W, bench.NOISE, nv12=True, out_fmt=L.FMT_U8_NHWC),
             "b": DenoiseUpscalePipeline(den, sr, H, W, bench.NOISE, nv12=True, out_fmt=L.FMT_NV12)}
    chunks = [bench.synth_nv12(ch.load_lo, ch.load_hi, dev, variant=v) for v in range(2)]
    outs = {m: p.new_output(F) for m, p in pipes.items()}
    nv_shape = pipes["b"].out_frame_shape()
    nv_a = torch.empty((F,) + nv_shape, dtype=torch.uint8, device=dev)

    def step(m, i):
        pipes[m].run(chunks[i % 2], ch.owned, outs[m])
        if m == "a":
            rgb_to_nv12_into(eng, outs["a"], nv_a)    # one launch over the step's frames

    # ---- correctness: both modes' NV12 frames, byte for byte
    step("a", 0)
    step("b", 0)
    torch.cuda.synchronize()
    identical = bool(torch.equal(nv_a, outs["b"]))

    # ---- device-resident frames/s, modes alternated
    for m in "ab":
        for i in range(args.warmup):
            step(m, i)
    torch.cuda.synchronize()
    dev_fps = {"a": [], "b": []}
    for r in range(args.repeats):
        for m in ("ab" if r % 2 == 0 else "ba"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                step(m, i)
            e1.record()
            torch.cuda.synchronize()
            dev_fps[m].append(F * args.steps / (e0.elapsed_time(e1) / 1000))

    # ---- host path: pinned NV12 chunk in -> pinned NV12 frames out
    chunks_host = [c.cpu().pin_memory() for c in chunks]
    host_fps = {"a": [], "b": []}
    steppers = {}
    for m in "ab":
        outs_host = [torch.empty((F,) + nv_shape, dtype=torch.uint8).pin_memory() for _ in range(2)]
        steppers[m] = host_step_factory(pipes[m], eng, chunks_host[0], ch.owned, outs_host, convert=(m == "a"))
        for i in range(2):
            steppers[m][0](i)
        steppers[m][1]()
    for r in range(args.repeats):
        for m in ("ab" if r % 2 == 0 else "ba"):
            st, sync = steppers[m]
            t0 = time.perf_counter()
            for i in range(args.steps):
                st(i)
            sync()
            host_fps[m].append(F * args.steps / (time.perf_counter() - t0))

    # ---- conv_last launch time (un-graphed profile runs, CUDA events between the steps)
    lr0 = torch.rand(1, 3, H, W, device=dev)
    conv_last = {}
    for m in "ab":
        p = pipes[m].sr_plan
        o = p.new_output()
        runs = [p.profile(lr0, o) for _ in range(args.profile_runs + 1)][1:]
        conv_last[m] = statistics.median(r[-1][0] for r in runs) * 1000
    conv_u8 = outs["a"][0:1]
    nv_kernel_us = bench.timed_kernel(lambda: rgb_to_nv12_into(eng, conv_u8, nv_a[0:1]), iters=50) * 1000

    med = {k: {m: statistics.median(v[m]) for m in "ab"} for k, v in (("dev", dev_fps), ("host", host_fps))}
    return {
        "metric": "NV12 output of cfg3: (a) uint8 RGB + ss4k_rgb_to_nv12 vs (b) out_fmt NV12",
        "card": card(), "n_gpus": 1, "frames_per_step": F, "steps": args.steps, "repeats": args.repeats,
        "out_frame": f"{2 * W}x{2 * H}",
        "bytes_per_frame": {"a_uint8_rgb": outs["a"][0].numel(), "a_nv12_after_conversion": nv_a[0].numel(), "b_nv12": outs["b"][0].numel()},
        "nv12_identical": identical,
        "device_fps": {"a": med["dev"]["a"], "b": med["dev"]["b"], "b_over_a": med["dev"]["b"] / med["dev"]["a"],
                       "runs_a": dev_fps["a"], "runs_b": dev_fps["b"]},
        "host_fps": {"a": med["host"]["a"], "b": med["host"]["b"], "b_over_a": med["host"]["b"] / med["host"]["a"],
                     "runs_a": host_fps["a"], "runs_b": host_fps["b"],
                     "note": "pinned NV12 chunk H2D -> nets -> per frame (a: rgb_to_nv12 ->) D2H of NV12 frames, copy stream overlapping the next frame"},
        "conv_last_us": {"a_uint8_store": conv_last["a"], "b_nv12_store": conv_last["b"],
                         "a_rgb_to_nv12_kernel_per_frame": nv_kernel_us,
                         "note": "median of %d un-graphed ss4k_plan_profile runs; the conversion kernel timed over 50 launches on one frame" % args.profile_runs},
    }


def _gather_worker(rank, world, F, H, W, steps, q):
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29517")
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    res = {}
    for name, shape in (("a_uint8_rgb", (F, 2 * H, 2 * W, 3)), ("b_nv12", (F, 3 * H, 2 * W))):
        local = torch.randint(0, 256, shape, dtype=torch.uint8, device=dev)
        bufs = [torch.empty_like(local) for _ in range(world)] if rank == 0 else None
        host = torch.empty((world,) + shape, dtype=torch.uint8).pin_memory() if rank == 0 else None
        times = []
        for i in range(steps + 2):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dist.gather(local, bufs, dst=0)
            if rank == 0:
                for r in range(world):
                    host[r].copy_(bufs[r], non_blocking=True)
            torch.cuda.synchronize()
            if i >= 2:
                times.append(1000 * (time.perf_counter() - t0))
        res[name] = {"ms_median": statistics.median(times), "bytes_to_rank0_host": world * local.numel()}
    if rank == 0:
        q.put(res)
    dist.barrier()
    dist.destroy_process_group()


def gather_two_gpus(args):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        return {"skipped": f"{torch.cuda.device_count()} GPU(s) visible"}
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, args.clip, bench.FRAME_H, bench.FRAME_W, args.steps, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
    res["note"] = "NCCL gather of one step's finished frames (clip frames per rank) to rank 0 + its D2H copy into pinned memory"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1, choices=[1, 2])
    ap.add_argument("--clip", type=int, default=8, help="owned frames per step")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=4, help="alternations of the two modes")
    ap.add_argument("--profile-runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_nv12_out.py needs a CUDA device")
    line = single_gpu(args)
    if args.gpus == 2:
        line["gather_2gpus"] = gather_two_gpus(args)
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
