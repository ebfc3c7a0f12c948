/*
 * ss4k.h -- C ABI of the B200-native (sm_100a) per-frame video enhancement engine.
 *
 * This is the drop-in boundary for ONE hot path of gmlwns2000/sharkshark-4k:
 * BSVD temporal denoiser -> RealESRGAN upscaler (RRDBNet x2/x4, SRVGGNetCompact).
 * The reference has no FFI of its own (it is pure Python over torch.nn.Conv2d -> cuDNN /
 * TensorRT), so every entry point below names the reference Python interface it
 * replaces.  All paths are relative to the reference tree.
 *
 *   ss4k_create / ss4k_destroy       engine life time == FsrcnnUpscalerService.proc_init /
 *                                    proc_cleanup      (src/upscale/fsrcnn_upscaler.py:118-142)
 *   ss4k_load_weights                state-dict load   (realesrgan/factory.py:160-170 via
 *                                    RealESRGANer; bsvd/model.py:487-499 BSVD.load)
 *   ss4k_plan_create                 build_model(...)  (realesrgan/factory.py:108-234,
 *                                    bsvd/factory.py:21-83): arch + shape -> compiled callable
 *   ss4k_run                         model(x)          (fsrcnn_upscaler.py:181,294 ; 277 for BSVD clip)
 *   ss4k_run_host                    same, with host (pinned) buffers: the copies the
 *                                    reference does in pipeline.py:91 (H2D) and streamer.py:95 (D2H)
 *   ss4k_bsvd_stream_*               BSVD.feedin_one_element / streaming_forward / reset
 *                                    (bsvd/model.py:510-513,526-580)
 *   ss4k_conv3x3                     one nn.Conv2d(k=3,p=1)+act (operator-level entry used by the
 *                                    kernel parity tests; every net is a sequence of these)
 *
 * Conventions
 *   - every function returns 0 on success, a negative SS4K_E_* code otherwise; nothing
 *     aborts, exits or throws across this boundary.  ss4k_last_error() gives the text.
 *   - the caller owns input/output buffers (device pointers + the CUDA stream they are
 *     valid on); the library owns weights, workspaces, CUDA graphs and BSVD ring buffers.
 *   - a context is bound to one device and used by one thread at a time.
 *   - there is NO CPU fallback: without a CUDA device of compute capability 10.x,
 *     ss4k_create fails with SS4K_E_NODEVICE.
 */
#ifndef SS4K_H_
#define SS4K_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SS4K_ABI_VERSION 1

/* error codes */
#define SS4K_OK 0
#define SS4K_E_INVALID (-1)   /* bad argument / unsupported configuration          */
#define SS4K_E_NODEVICE (-2)  /* no sm_100 device / CUDA driver not usable         */
#define SS4K_E_CUDA (-3)      /* a CUDA runtime / driver call failed               */
#define SS4K_E_WEIGHTS (-4)   /* a weight tensor is missing or has the wrong shape */
#define SS4K_E_SELFTEST (-5)  /* tcgen05 descriptor self-probe found no working mode */
#define SS4K_E_NOMEM (-6)

/* network architectures (reference: realesrgan/factory.py:112-138, bsvd/factory.py:31-35) */
#define SS4K_ARCH_SRVGG 0 /* SRVGGNetCompact(num_feat=64, num_conv, upscale, prelu) */
#define SS4K_ARCH_RRDB 1  /* basicsr RRDBNet(num_feat=64, num_block, num_grow_ch=32, scale) */
#define SS4K_ARCH_BSVD 2  /* BSVD(chns=[32,64,128], mid_ch=32, interm_ch=30, relu6, norm none) */

/* element types of weight tensors handed to ss4k_load_weights */
#define SS4K_DT_F32 0
#define SS4K_DT_F16 1

/* arithmetic mode of the tensor-core path (operands; accumulation is always fp32) */
#define SS4K_ACT_F16 0        /* fp16 operands, fp16 activations in HBM (default)       */
#define SS4K_ACT_BF16 1       /* bf16 operands                                          */
#define SS4K_ACT_F16_SPLIT 2  /* fp16 hi/lo split operands, 3 MMAs per product (BSVD
                                 with the reference constructor's kaiming init)        */

/* frame formats at the boundary */
#define SS4K_FMT_F32_NCHW 0 /* float [N,3,H,W] in [0,1]   (model(x) boundary)          */
#define SS4K_FMT_F16_NCHW 1
#define SS4K_FMT_U8_NHWC 2  /* uint8 [N,H,W,3]            (upscale(frames) boundary)   */
#define SS4K_FMT_NV12 3     /* Y plane u8[H,W] + interleaved UV u8[H/2,W] per frame    */

typedef struct ss4k_ctx ss4k_ctx;
typedef struct ss4k_plan ss4k_plan;
typedef struct ss4k_bsvd_stream ss4k_bsvd_stream;

typedef struct ss4k_plan_cfg {
  int32_t struct_size; /* = sizeof(ss4k_plan_cfg), for ABI growth */
  int32_t net_id;      /* weight slot filled by ss4k_load_weights             */
  int32_t arch;        /* SS4K_ARCH_*                                         */
  int32_t n, h, w;     /* input batch / frame size (BSVD: n = frames of the clip) */
  int32_t scale;       /* SRVGG: upscale; RRDB: 2 or 4; BSVD: ignored         */
  int32_t depth;       /* SRVGG: num_conv (16/32); RRDB: num_block (23/6); BSVD: ignored */
  int32_t tile;        /* RealESRGANer tile (0 = off), tile_pad as in ArgsData (factory.py:93-95) */
  int32_t tile_pad;
  int32_t act_mode;    /* SS4K_ACT_*                                          */
  int32_t in_fmt;      /* SS4K_FMT_*                                          */
  int32_t out_fmt;     /* SS4K_FMT_* (U8: clamp to [0,1], *255, truncate like fsrcnn_upscaler.py:233).
                        * NV12 (SS4K_ARCH_RRDB only; SRVGG and BSVD plans return SS4K_E_INVALID): packed frames
                        * [n, oh*3/2, ow] bytes, the Y plane u8[oh,ow] then interleaved UV u8[oh/2,ow] per frame (the layout
                        * in_fmt SS4K_FMT_NV12 and ss4k_nv12_unpack use); oh % 2 == 0 and ow % 4 == 0 are required.  The
                        * result is bit-identical to ss4k_rgb_to_nv12 applied to the same plan's SS4K_FMT_U8_NHWC output.
                        * Untiled plans convert in the last convolution's epilogue; tiled plans (and a last convolution
                        * off the streaming kernel) write uint8 RGB into a frame of the plan and convert it in a step of
                        * its own. */
  int32_t use_graph;   /* 1: capture the per-frame launch sequence in a CUDA graph */
  int32_t reserved[8]; /* [1]: RealESRGANer pre_pad (factory.py:95): reflect pad on the right / bottom before tiling, cropped
                        *      off the output; the x2 nets also get RealESRGANer's reflect mod-2 pad for odd sizes.  tile,
                        *      tile_pad, pre_pad are applied INSIDE the plan: crops of one shape run as one batch.
                        * [0]: BSVD with a 3-channel frame format (SS4K_FMT_U8_NHWC / SS4K_FMT_NV12): bit pattern of the
                        * float noise level written into the 4th input channel (0.1 * denoise_rate,
                        * fsrcnn_upscaler.py:262); with the float / half NCHW formats the caller supplies 4 channels */
} ss4k_plan_cfg;

/* engine ------------------------------------------------------------------------------- */
int ss4k_abi_version(void);
int ss4k_create(int device_id, ss4k_ctx** out_ctx);
int ss4k_destroy(ss4k_ctx* ctx);
const char* ss4k_last_error(ss4k_ctx* ctx); /* ctx may be NULL: error of the failed ss4k_create */
/* which tcgen05 shared-memory-descriptor addressing mode the start-up self-probe selected
 * (0: shifted start address; 1: shifted start address + base_offset; 2: one TMA box per tap column) */
int ss4k_desc_mode(ss4k_ctx* ctx);
int ss4k_set_desc_mode(ss4k_ctx* ctx, int mode);
/* number of kernel launches issued by this context so far (bench.py "gpu_launches") */
int64_t ss4k_launch_count(ss4k_ctx* ctx);

/* weights ------------------------------------------------------------------------------ */
/* name = state-dict key ("body.0.weight", "conv_first.bias", "temp1.inc.convblock.0.weight", ...);
 * host_ptr = contiguous tensor of `dtype`, shape[ndim] as in the state dict (conv: OIHW). */
int ss4k_load_weights(ss4k_ctx* ctx, int net_id, const char* name, const void* host_ptr,
                      int dtype, const int64_t* shape, int ndim);
int ss4k_clear_weights(ss4k_ctx* ctx, int net_id);

/* plans -------------------------------------------------------------------------------- */
int ss4k_plan_create(ss4k_ctx* ctx, const ss4k_plan_cfg* cfg, ss4k_plan** out_plan);
int ss4k_plan_destroy(ss4k_plan* plan);
/* output geometry of a plan: n, c, h, w of the result image (NV12 output: still (n, 3, oh, ow); the buffer holds
 * n * oh * ow * 3 / 2 bytes, as ss4k_plan_io_bytes reports) */
int ss4k_plan_out_shape(const ss4k_plan* plan, int32_t out_nchw[4]);
/* algorithmic FLOPs of one ss4k_run (2*Cin*Cout*9*Hout*Wout summed over convs, true channel counts) */
double ss4k_plan_flops(const ss4k_plan* plan);
/* number of kernel launches (graph nodes included) one ss4k_run issues */
int ss4k_plan_launches(const ss4k_plan* plan);
/* how many of those steps replay from the plan's CUDA graph (0: graph capture unavailable / disabled) */
int ss4k_plan_graph_steps(const ss4k_plan* plan);
/* steps of the layer program (== entries ss4k_plan_profile returns; every step is one launch, except a layout step whose
 * work the first conv's loader does, which launches nothing) */
int ss4k_plan_steps(const ss4k_plan* plan);
/* JSON description of the layer program (buffers, convs, epilogues); malloc'd, free with ss4k_free.
 * Works without a GPU when the plan was built with ss4k_plan_dry (host-side planner only). */
int ss4k_plan_dry(const ss4k_plan_cfg* cfg, char** out_json);
void ss4k_free(void* p);

/* run: device pointers valid on `cuda_stream` (a cudaStream_t / CUstream passed as void*) */
int ss4k_run(ss4k_plan* plan, const void* in_dev, void* out_dev, void* cuda_stream);
/* run with host buffers (pinned or pageable): H2D copy, run, D2H copy, stream-ordered on an
 * internal stream; returns after the result is in out_host. */
int ss4k_run_host(ss4k_plan* plan, const void* in_host, void* out_host);
/* the same as a software pipeline over successive frames (the reference's producer / consumer queues,
 * src/sharkshark/pipeline.py:61-138): the call returns once the work is queued; the H2D copy of call i+1 and the D2H
 * copy of call i-1 overlap the kernels of call i (two device staging slots, copy streams of their own).  in_host /
 * out_host (pinned) must stay valid, and out_host unread, until ss4k_plan_host_sync returns; at most two calls'
 * out_host buffers are in flight, so alternate between two. */
int ss4k_run_host_async(ss4k_plan* plan, const void* in_host, void* out_host);
int ss4k_plan_host_sync(ss4k_plan* plan);
/* bytes of one run's input / output buffer in the plan's in_fmt / out_fmt (NV12: n * h * w * 3 / 2); ss4k_run_host and
 * ss4k_run_host_async copy exactly these sizes */
int ss4k_plan_io_bytes(const ss4k_plan* plan, int64_t* in_bytes, int64_t* out_bytes);
/* measurement entry (bench.py roofline): one run of the plan without its CUDA graph, a CUDA event between
 * every step on `cuda_stream`.  ms[i] = device time of step i, flops[i] = its algorithmic FLOPs,
 * kind[i] = 0 layout/colour kernel, 1 row-streaming conv kernel, 2 tile conv kernel, 4 a layout step done by the
 * first conv's loader (no launch of its own).  An NV12-output plan whose last conv does not store NV12 itself has
 * one more step at the end: the uint8 RGB -> NV12 conversion (kind 0).  Returns the step count (<= cap) or a negative
 * error. */
int ss4k_plan_profile(ss4k_plan* plan, const void* in_dev, void* out_dev, void* cuda_stream, float* ms,
                      double* flops, int32_t* kind, int cap);

/* colour stage on the encoder side (north star part 4; the reference hands rgb24 to an ffmpeg pipe,
 * src/stream/twitch_stream/output_stream.py:115-175, and lets swscale convert): uint8 NHWC RGB frames
 * [n,h,w,3] -> NV12 (Y plane u8[h,w] + interleaved UV u8[h/2,w] per frame), BT.709 limited range, 15-bit fixed
 * point, chroma = mean of the 2x2 block.  h % 2 == 0, w % 4 == 0.  Device pointers. */
int ss4k_rgb_to_nv12(ss4k_ctx* ctx, const void* rgb_dev, void* nv12_dev, int n, int h, int w, void* cuda_stream);

/* ingest / egress surfaces (SURVEY.md section 8f N3).  A hardware decoder hands out, and a hardware encoder takes, PITCHED
 * NV12 device surfaces, one allocation per frame: luma rows `pitch` bytes apart, the interleaved chroma plane at its own
 * pointer (cuvidMapVideoFrame: base + pitch * coded_height; NvEncRegisterResource: base + pitch * height).  These two
 * entries move n such surfaces into / out of the packed frame chunk the plans read (in_fmt SS4K_FMT_NV12:
 * [n, h*3/2, w] bytes) with 2-D DMA copies on `cuda_stream` -- no kernel, no host round trip.  They replace the rgb24 OS
 * pipes of src/stream/twitch_realtime_handler/twitchgrabber.py:91-102 and src/stream/twitch_stream/output_stream.py:115-191.
 * `surfaces` is a HOST array; all pointers in it are device pointers. */
typedef struct ss4k_nv12_surface {
  void* y;             /* luma plane: h rows of w bytes, pitch_y bytes apart                    */
  void* uv;            /* interleaved chroma plane: h/2 rows of w bytes, pitch_uv bytes apart   */
  int32_t pitch_y, pitch_uv;
} ss4k_nv12_surface;
int ss4k_nv12_pack(ss4k_ctx* ctx, const ss4k_nv12_surface* surfaces, int n, int h, int w, void* packed_dev, void* cuda_stream);
int ss4k_nv12_unpack(ss4k_ctx* ctx, const void* packed_dev, const ss4k_nv12_surface* surfaces, int n, int h, int w, void* cuda_stream);

/* BSVD streaming (persistent per-stream ring buffers) ----------------------------------- */
/* open: plan must be an SS4K_ARCH_BSVD plan (its n is ignored; frames are pushed one at a time).  Every precision mode
 * streams (split precision: every ring has a low-half twin).  Ring lengths are powers of two, so a steady-state push (all
 * layers active, no clip boundary in reach) replays one captured CUDA graph per phase of the longest ring between a copy
 * into and a copy out of stream-owned staging buffers (plan cfg use_graph = 0 or SS4K_NO_STREAM_GRAPH: per-layer launches). */
int ss4k_bsvd_stream_open(ss4k_plan* plan, ss4k_bsvd_stream** out_stream);
/* like ss4k_bsvd_stream_open, for pushes of up to max_frames (>= 1) frames per call.  Every conv of the streaming kernel
 * then runs once over the frames of a push, its ring slots wrapping inside the kernel.  Each ring holds max_frames - 1
 * more frames (lengths still rounded up to powers of two); max_frames = 1 is ss4k_bsvd_stream_open.  Steady-state
 * pushes replay one graph per (phase, frame count). */
int ss4k_bsvd_stream_open_batched(ss4k_plan* plan, int max_frames, ss4k_bsvd_stream** out_stream);
/* push frame t (in_dev: one frame in the plan's in_fmt: 4 channels RGB + noise map for the float / half NCHW formats, a
 * uint8 RGB or NV12 frame for the frame formats -- the noise map is then the plan's reserved[0] level).
 * *got_output = 1 when the denoised frame t-16 was written to out_dev (3 channels). */
int ss4k_bsvd_stream_push(ss4k_bsvd_stream* s, const void* in_dev, void* out_dev,
                          int* got_output, void* cuda_stream);
/* push frames t .. t+n-1 (1 <= n <= max_frames; in_dev: n frames back to back in the plan's in_fmt); out_dev has room for
 * n frames of 3 channels; *n_out = number of denoised frames written, oldest first (frames t-16 .. t+n-17 that exist).
 * n outside [1, max_frames], a null pointer or a push after flush without reset: SS4K_E_INVALID. */
int ss4k_bsvd_stream_push_frames(ss4k_bsvd_stream* s, const void* in_dev, int n, void* out_dev, int* n_out, void* cuda_stream);
/* flush: feed "None" (end-of-clip) steps until the next denoised frame falls out of the pipeline;
 * call until *got_output == 0 (all frames of the clip delivered; one frame per call, whatever the pushes carried) */
int ss4k_bsvd_stream_flush(ss4k_bsvd_stream* s, void* out_dev, int* got_output, void* cuda_stream);
int ss4k_bsvd_stream_reset(ss4k_bsvd_stream* s);
/* frames of latency between a push and its output (BSVD.count_shift, model.py:582-588: 16) */
int ss4k_bsvd_stream_latency(const ss4k_bsvd_stream* s);
int ss4k_bsvd_stream_close(ss4k_bsvd_stream* s);

/* service glue (fsrcnn_upscaler.py:168-326): HBM-bound statistics / pooling / stencil / finalising kernels -------- */
/* image formats: 0 float NCHW, 1 half NCHW, 2 uint8 NHWC (read as value/255).  All pointers are DEVICE pointers. */
/* per-(n,c) sum and sum of squares (double[n*c][2]); replaces .mean()/.std() of fsrcnn_upscaler.py:191-196,305-310 */
int ss4k_glue_chan_stats(const void* img, int fmt, int n, int c, int h, int w, double* sums_dev, void* cuda_stream);
/* F.interpolate(mode='area') -> float NCHW [n,c,oh,ow]  (fsrcnn_upscaler.py:174-176,204-209,239-241);
 * SS4K_E_INVALID unless n, c, h, w, oh, ow >= 1 */
int ss4k_glue_area_pool(const void* img, int fmt, int n, int c, int h, int w, float* out_dev, int oh, int ow,
                        void* cuda_stream);
/* low-res colour difference blur_k(a*hb + b - lb), reflect padding (fsrcnn_upscaler.py:211-213); a, b = the
 * distribution-match affine map derived from the sums (NULL sums: a=1, b=0).  SS4K_E_INVALID unless ksize is odd and
 * positive, ksize/2 < h, ksize/2 < w (the limits of the reference's F.pad(mode='reflect')), n >= 1 and c >= 1 */
int ss4k_glue_blur_diff(const float* hb, const float* lb, float* diff, const float* kern_dev, int ksize, int n, int c,
                        int h, int w, const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr,
                        void* cuda_stream);
/* clamp(a*hr + b - bilinear_up(diff), 0, 1) -> uint8 NHWC (truncating unless round_u8) or float NCHW
 * (fsrcnn_upscaler.py:197-198,214-220,232-233); diff may be NULL, otherwise dh >= 1 and dw >= 1 (SS4K_E_INVALID) */
int ss4k_glue_finalize(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                       const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* out_u8,
                       float* out_f32, int round_u8, void* cuda_stream);
/* F.interpolate(mode='bicubic') of a float NCHW image, clamp, uint8 NHWC (fsrcnn_upscaler.py:222-233) */
/* finalize + bicubic resize + uint8 in one pass (no full-resolution fp32 intermediate): the tail of upscale_multi /
 * upscale_single when output_shape differs from the net's output (fsrcnn_upscaler.py:214-233,315-326).  c == 3;
 * downscale factors up to about 2 (h/oh * 7 + 5 <= 24 and w/ow * 31 + 5 <= 72); diff NULL or dh, dw >= 1 */
int ss4k_glue_finalize_bicubic_u8(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                                  const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr,
                                  uint8_t* out_u8, int oh, int ow, int round_u8, void* cuda_stream);
/* the two entries above with NV12 output for an encoder: packed frames [n, oh*3/2, ow] (Y plane u8[oh,ow], then
 * interleaved UV u8[oh/2,ow]; the layout of in_fmt SS4K_FMT_NV12 and ss4k_nv12_unpack).  The bytes are exactly those of
 * the uint8 entry with the same arguments (same truncation or round_u8 rounding) followed by ss4k_rgb_to_nv12 (BT.709
 * limited range, 15-bit fixed point, chroma = mean of the 2x2 block), without the uint8 RGB frame.  SS4K_E_INVALID
 * unless c == 3, the output height is even, the output width is a multiple of 4 and out_nv12 is 4-byte aligned; the
 * geometry checks of the uint8 entries (diff sizes, the patch guard of the resizing form) apply unchanged.
 * finalize_nv12: no resize, the output is (h, w); h, w, n >= 1. */
int ss4k_glue_finalize_nv12(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                            const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr,
                            uint8_t* out_nv12, int round_u8, void* cuda_stream);
int ss4k_glue_finalize_bicubic_nv12(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                                    const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr,
                                    uint8_t* out_nv12, int oh, int ow, int round_u8, void* cuda_stream);
/* SS4K_E_INVALID unless n, c, h, w, oh, ow >= 1 */
int ss4k_glue_bicubic_u8(const float* in, int n, int c, int h, int w, uint8_t* out, int oh, int ow, int round_u8,
                         void* cuda_stream);
/* opacity * clamp(sharpen_ker(strength)(x), 0, 1) + (1-opacity) * other -> float NCHW; other may be NULL
 * (fsrcnn_upscaler.py:54-84,278-281,298-299).  SS4K_E_INVALID for h < 2 or w < 2 (3x3 reflect padding) */
int ss4k_glue_sharpen_blend(const void* x, int fmt, int n, int c, int h, int w, float strength, float opacity,
                            const void* other, int other_fmt, float* out, void* cuda_stream);
/* the same, written as an upscaler plan's first-layer activation tensor (ss4k_plan_input_act: 16-bit NHWC, channel
 * pitch `pitch`, pixel_unshuffle(`unshuffle`) channel order): the denoise -> upscale hand-over of upscale_single
 * (fsrcnn_upscaler.py:278-295) without a float image and without a layout kernel in front of conv_first.
 * SS4K_E_INVALID for h < 2 or w < 2, h or w not a multiple of unshuffle, pitch not a multiple of 8 or below
 * c * unshuffle^2 */
int ss4k_glue_sharpen_blend_act(const void* x, int fmt, int n, int c, int h, int w, float strength, float opacity,
                                const void* other, int other_fmt, void* act_out, int unshuffle, int pitch, int is_bf16,
                                void* cuda_stream);
/* device pointer / layout of the tensor a plan's layout step writes (fails for tiled, split-precision and frame-decoding
 * plans, which have no plain layout step), and ss4k_run without that step: the caller has filled the tensor itself */
int ss4k_plan_input_act(ss4k_plan* plan, void** act_dev, int32_t* pitch, int32_t* unshuffle, int32_t* is_bf16);
int ss4k_run_act(ss4k_plan* plan, void* out_dev, void* cuda_stream);

/* host-only: the tile grid of a plan configuration (tile, tile_pad, reserved[1] = pre_pad) and its packing into crop
 * atlases as JSON; free with ss4k_free */
int ss4k_debug_tile_layout(const ss4k_plan_cfg* cfg, char** out_json);
/* host-only: a BSVD stream's layout for pushes of up to max_frames frames as JSON -- shift_num, period, every buffer's
 * ring length and producer lag, every step's lag, buffers read / written and whether it scatters (temporal shift); free
 * with ss4k_free */
int ss4k_debug_bsvd_stream_layout(const ss4k_plan_cfg* cfg, int max_frames, char** out_json);

/* operator-level entry (kernel parity tests) -------------------------------------------- */
typedef struct ss4k_conv_desc {
  int32_t struct_size;
  int32_t n, h, w;        /* input geometry                                         */
  int32_t cin, cout;
  int32_t mode;           /* 0: 3x3 s1 p1; 1: nearest-x2 upsample then 3x3 s1 p1; 2: 3x3 s2 p1 */
  int32_t act;            /* 0 none, 1 PReLU/LeakyReLU (slope[cout]), 2 ReLU6        */
  int32_t act_mode;       /* SS4K_ACT_*                                              */
  int32_t pixel_shuffle;  /* 0, or r: output is PixelShuffle(r) of the conv result   */
  float alpha;            /* out = alpha*act(conv+bias) + beta*residual              */
  float beta;
  int32_t reserved[8];
} ss4k_conv_desc;
/* x: float NCHW [n,cin,h,w]; weight OIHW float; bias[cout]; slope[cout] or NULL;
 * residual: float NCHW of the output shape or NULL; y: float NCHW output.  All DEVICE pointers.
 * Internally: convert to fp16 NHWC, run the tcgen05 kernel, convert back. */
int ss4k_conv3x3(ss4k_ctx* ctx, const ss4k_conv_desc* d, const float* x, const float* weight,
                 const float* bias, const float* slope, const float* residual, float* y,
                 void* cuda_stream);

/* host-only debug entry (no GPU needed): packed weight layout + MMA schedule of one conv, used by the
 * CPU tests that emulate the kernel schedule.  out_json / out_packed are malloc'd: ss4k_free. */
int ss4k_debug_pack(const ss4k_conv_desc* d, int in_pitch, int in_coff, int wperm, const float* w_host,
                    const float* bias_host, const float* slope_host, char** out_json, float** out_packed,
                    int64_t* out_count);

/* profiling entry: average milliseconds of one launch of the described conv over `iters` launches
 * (CUDA events on the context's stream).  dbg_flags: 1 skip MMA issue, 2 skip TMA loads, 4 skip epilogue
 * math/stores (pipeline experiments; results are then meaningless).  out_json (optional): tile config. */
int ss4k_debug_bench_conv(ss4k_ctx* ctx, const ss4k_conv_desc* d, int slab_pitch, int dbg_flags, int iters,
                          float* ms_per_launch, char** out_json);

#ifdef __cplusplus
}
#endif
#endif /* SS4K_H_ */
