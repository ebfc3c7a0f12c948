"""Small end-to-end runs for compute-sanitizer (memcheck): SRVGG, RRDBNet (dense slab, residual epilogues, TMA stores),
BSVD clip (stride-2 tile kernel, scatter stores, split mode)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import ss4k_b200
from ss4k_b200 import _lib as L, realesrgan, bsvd as nb
from oracle import rrdbnet, srvgg, bsvd as ob
torch.manual_seed(0)
x = torch.rand(1, 3, 24, 136).cuda()
m = realesrgan.NativeSRVGG(srvgg.SRVGGNetCompact(3, 3, 64, 2, 4).eval().state_dict(), num_conv=2, upscale=4, device=0, use_graph=False)
print("srvgg", tuple(m(x).shape))
m = realesrgan.NativeRRDBNet(rrdbnet.RRDBNet(3, 3, 2, 64, 1, 32).eval().state_dict(), scale=2, num_block=1, device=0, use_graph=False)
print("rrdb", tuple(m(x).shape))
for mode in (L.ACT_F16, L.ACT_F16_SPLIT):
    d = nb.NativeBSVD(ob.build_bsvd32(0, weight_scale=0.5), device=0, act_mode=mode, use_graph=False)
    print("bsvd", mode, tuple(d(torch.rand(1, 2, 4, 16, 136).cuda()).shape))
# uint8 frames in / out (packed RGB row stores, ragged width), and the service glue with the SRVGG half-NCHW PixelShuffle store
net = rrdbnet.RRDBNet(3, 3, 2, 64, 1, 32).eval()
m = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=1, device=0, use_graph=False)
fr = torch.randint(0, 256, (1, 24, 150, 3), dtype=torch.uint8).cuda()
print("rrdb u8", tuple(m._plan(1, 24, 150, L.FMT_U8_NHWC, L.FMT_U8_NHWC).run(fr).shape))
from ss4k_b200 import service
sv = service.FsrcnnUpscalerService(lr_level=0, device=0, denoising=False, model_name='realesr-animevideov3',
                                   state_dict=srvgg.SRVGGNetCompact(3, 3, 64, 16, 4).eval().state_dict())
sv.proc_init()
sv.output_shape = (130, 270)
print("service", tuple(sv.upscale(torch.randint(0, 256, (1, 72, 136, 3), dtype=torch.uint8).cuda()).shape))
sv.output_shape = None
print("service", tuple(sv.upscale(torch.randint(0, 256, (1, 72, 136, 3), dtype=torch.uint8).cuda()).shape))
print("rgb->nv12", tuple(ss4k_b200.Engine.get(0).rgb_to_nv12(torch.randint(0, 256, (1, 8, 32, 3), dtype=torch.uint8).cuda()).shape))
# NV12 output of the service glue: the fused finalise + bicubic store (ragged 32 x 8 tiles: 150 rows, 280 columns) and the
# no-resize finalise store (ragged width), into buffers of exactly the frames' size
sv.out_fmt = L.FMT_NV12
sv.output_shape = (150, 280)
print("service nv12", tuple(sv.upscale(torch.randint(0, 256, (2, 72, 136, 3), dtype=torch.uint8).cuda()).shape))
sv.output_shape = None
print("service nv12", tuple(sv.upscale(torch.randint(0, 256, (1, 18, 35, 3), dtype=torch.uint8).cuda()).shape))
# round 2: frame decode in the first BSVD conv (decoder warps, NV12 and uint8 RGB, ragged width, owned range), split
# precision twin-tile stores and specialised store paths, ring-buffer streaming (split, phase graphs), the cfg3 pipeline
# with the glue writing the upscaler's first activation tensor, in-engine tiling, NV12 surfaces
from ss4k_b200.pipeline import DenoiseUpscalePipeline
for mode in (L.ACT_F16, L.ACT_F16_SPLIT):
    d = nb.NativeBSVD(ob.build_bsvd32(0, weight_scale=0.5), device=0, act_mode=mode, use_graph=False)
    nv = torch.randint(16, 236, (5, 36, 136), dtype=torch.uint8).cuda()
    print("bsvd nv12", mode, tuple(d.denoise_frames(nv.reshape(5, -1), 24, 136, 0.075, nv12=True, own=(1, 4)).shape))
    rgb = torch.randint(0, 256, (3, 24, 264, 3), dtype=torch.uint8).cuda()
    print("bsvd u8", mode, tuple(d.denoise_frames(rgb, 24, 264, 0.075).shape))
    st = d.stream(16, 136)
    xs = torch.rand(40, 4, 16, 136).cuda()
    outs = [o for o in (st.push(xs[i]) for i in range(40)) if o is not None] + list(st.flush())
    st.close()
    print("bsvd stream", mode, len(outs))
den = nb.NativeBSVD(ob.build_bsvd32(0), device=0, act_mode=L.ACT_F16_SPLIT, out_dtype=torch.float16)
pipe = DenoiseUpscalePipeline(den, m, 24, 136, 0.075, nv12=True)
print("cfg3", tuple(pipe.run(torch.randint(16, 236, (4, 36 * 136), dtype=torch.uint8).cuda(), slice(1, 3)).shape))
mt = realesrgan.NativeRRDBNet(net.state_dict(), scale=2, num_block=1, device=0, use_graph=False, tile=32, tile_pad=6, pre_pad=3)
print("tiled", tuple(mt(torch.rand(1, 3, 45, 71).cuda()).shape))
eng = ss4k_b200.Engine.get(0)
pool = [torch.zeros(24, 64, dtype=torch.uint8, device="cuda") for _ in range(2)]
surf = [(p[:8, :40], p[16:20, :40]) for p in pool]
eng.nv12_unpack(torch.randint(0, 255, (2, 12, 40), dtype=torch.uint8).cuda(), surf, 8, 40)
print("surfaces", tuple(eng.nv12_pack(surf, 8, 40).shape))
torch.cuda.synchronize()
print("done")
