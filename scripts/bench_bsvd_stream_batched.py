"""BSVD ring-buffer streaming at 1280x720 with several frames per push (ss4k_bsvd_stream_push_frames): ms per frame in
steady state for n = 1, 2, 4, 8 frames per push, NV12 frames in, fp16 and split precision, one graph launch per push
(default) and per-layer launches (SS4K_NO_STREAM_GRAPH=1).  CUDA events around 96 frames after 64 frames of warm-up
(pipeline filled, every (phase, n) graph captured).  Prints the card's name and power limit first."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import ss4k_b200
from ss4k_b200 import _lib as L
from ss4k_b200 import bsvd as nbsvd
from oracle import bsvd as obsvd

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None}))

H, W, WARM, N = 720, 1280, 64, 96
frames = torch.randint(16, 236, (8, H * 3 // 2, W), dtype=torch.uint8, device="cuda")
for split in (False, True):
    sd = obsvd.build_bsvd32(0, weight_scale=1.0 if split else 0.5)
    den = nbsvd.NativeBSVD(sd, device=0, act_mode=L.ACT_F16_SPLIT if split else L.ACT_F16)
    for graph in (True, False):
        if graph:
            os.environ.pop("SS4K_NO_STREAM_GRAPH", None)
        else:
            os.environ["SS4K_NO_STREAM_GRAPH"] = "1"
        for n in (1, 2, 4, 8):
            s = den.stream(H, W, in_fmt=L.FMT_NV12, noise=0.075, max_frames=n)
            for i in range(WARM // n):
                s.push_frames(frames[:n])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for i in range(N // n):
                s.push_frames(frames[:n])
            e1.record()
            host_ms = (time.perf_counter() - t0) * 1000 / N
            torch.cuda.synchronize()
            print(json.dumps({"precision": "split" if split else "f16", "one_graph_per_push": graph, "frames_per_push": n,
                              "gpu_ms_per_frame": round(e0.elapsed_time(e1) / N, 3), "host_ms_per_frame": round(host_ms, 3)}),
                  flush=True)
            s.close()
