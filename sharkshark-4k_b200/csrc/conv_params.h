// Parameter block of the tcgen05 implicit-GEMM 3x3 convolution kernel (conv_tc.cu).
// Shared between the kernel and the host-side planner (engine.cpp).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ss4k {

constexpr int kTileW = 128;        // output pixels per tile row == UMMA M
constexpr int kBoxW = 130;         // halo row: kTileW + 2 pixels, one TMA box
constexpr int kRowBytes = 128;     // 64 channels * 2 bytes == one swizzle-128B row
constexpr int kMaxKBlocks = 12;
constexpr int kMaxTaps = 16;
constexpr int kMaxASlots = 8;
constexpr int kTmemCols = 512;
constexpr int kAccStageCols = 256; // two accumulator stages of 256 columns
constexpr int kSmemBytes = 232448; // 227 KB opt-in dynamic shared memory
constexpr int kConvThreads = 192;  // warp0 TMA, warp1 MMA, warps2-5 epilogue

// convolution "mode" == MMA schedule (see DESIGN.md section 4)
enum ConvMode : int {
  kModeConv3 = 0,  // 3x3 stride 1 pad 1: 9 taps
  kModeUp2 = 1,    // nearest-x2 upsample fused: 4 output phases x 4 pre-summed taps
  kModeS2 = 2      // 3x3 stride 2 pad 1 read through a (2C, W/2, 2, H/2, N) view: 4 taps, k-step masks
};

enum OutMode : int {
  kOutNHWC = 0,       // fp16/bf16 NHWC at (oy, ox), channel offset out_coff
  kOutNCHWF32 = 1,    // float NCHW, first `cout` channels (final conv)
  kOutPSNCHWF32 = 2,  // PixelShuffle(ps_r) into float NCHW (+ nearest-upsampled base image)  [SRVGG tail]
  kOutPS2NHWC = 3,    // PixelShuffle(2) into NHWC (weights' output channels pre-permuted to (a,b,c))
  kOutScatterNHWC = 4,// BSVD temporal shift: channel slices go to the t-1 / t+1 / t ring slots
  kOutNCHWF16 = 5,
  kOutU8NHWC = 6,     // clamp [0,1], *255, truncate or round, uint8 NHWC (3 channels)
  kOutPSNCHWF16 = 7,  // like kOutPSNCHWF32 with a half-precision destination
  kOutNV12 = 8        // the kOutU8NHWC bytes converted to NV12 (Y plane + interleaved UV per frame, BT.709 limited range,
                      // rgb_to_nv12_kernel's arithmetic): streaming kernel, NOUT == 16, cout == 3 only (conv_stream.cu)
};

enum ActKind : int { kActNone = 0, kActPRelu = 1, kActRelu6 = 2 };

struct KBlock {
  int32_t tmap;   // which activation tensor map (0: hi / only, 1: lo half of a split tensor)
  int32_t c0;     // first channel of this 64-channel block inside the source tensor
  int32_t p;      // coordinate in the "row phase" dimension (stride-2 view), else 0
  int32_t pad;
};

struct Tap {
  int8_t dr;      // input row of the tile this tap reads, relative to the output row (0..2)
  int8_t shift;   // pixel shift inside the halo row (0..2)
  int8_t sub;     // accumulator sub-index (output phase for kModeUp2), else 0
  int8_t pad;
};

struct Epilogue {
  const float* bias;     // [npad_total]
  const float* slope;    // [npad_total] negative-side slope (PReLU / LeakyReLU), or nullptr
  int32_t act;           // ActKind
  int32_t out_mode;      // OutMode
  float alpha;           // out = alpha*act(acc+bias) + beta1*res1 + beta2*res2
  float beta1, beta2;
  int32_t is_bf16;
  const void* res1;      // NHWC 16-bit, indexed at the OUTPUT pixel
  const void* res2;
  int32_t res1_pitch, res1_coff, res2_pitch, res2_coff;
  void* out;             // destination (see OutMode)
  void* out_lo;          // split mode: low halves (NHWC), or nullptr
  void* out2;            // scatter: slot receiving channels [0, fold)      (frame t-1's view)
  void* out3;            // scatter: slot receiving channels [fold, 2 fold) (frame t+1's view)
  int32_t out_pitch, out_coff;
  int32_t out_h, out_w;  // output image size (pixels)
  int32_t cout;          // real output channels of the whole conv
  int32_t ps_r;          // PixelShuffle factor for kOutPSNCHWF32
  int32_t fold;          // scatter fold (C/8)
  int32_t round_u8;      // kOutU8NHWC: 1 = round to nearest, 0 = truncate (fsrcnn_upscaler.py:233)
  const void* base;      // kOutPSNCHWF32: NHWC 16-bit base image (input of the net), pitch base_pitch
  int32_t base_pitch;
  int32_t res_sub;       // 1: residuals are indexed at output pixel, 0 same (kept for clarity)
  float slope_const;     // negative-side slope used when `slope` is null (LeakyReLU)
  int32_t res1_nch;      // > 0: only the first res1_nch channels of res1 are added (BSVD none_minus, model.py:436-442)
  // BSVD temporal shift (model.py:43-52) as channel-sliced STORES: when fold > 0 and out_mode is NHWC / PS2-NHWC,
  // output channels [0, fold) of frame t go to the tensor of frame t-1 (its "X_{t+1}[:fold]" input slice), channels
  // [fold, 2 fold) to frame t+1, the rest to frame t; slices that fall outside the clip are dropped (zero features).
  int64_t off_prev, off_next;  // element offsets from frame t's tensor to frame t-1's / t+1's
  int32_t t0, t_count;         // frame index of image n = 0 of this launch, clip length
  int64_t res1_lo_off, res2_lo_off;  // split mode: element offset of the residual's low halves (0: none)
  int32_t up2_store;     // 1: NHWC output is the nearest-x2 upsampled image: every pixel is stored at (2y+a, 2x+b), a, b in {0,1}
                         //    (out_h / out_w stay the conv's own grid; the destination tensor is 2*out_h x 2*out_w)
};

struct ConvParams {
  CUtensorMap tmA[2];    // activations, 5-D (C, W, P, H, N), box (64, box_w, 1, 1, 1), swizzle 128B
  CUtensorMap tmW;       // packed weights, 3-D (64, npad_total, nkb*ntaps), box (64, n_cta, ntaps)
  Epilogue ep;
  KBlock kb[kMaxKBlocks];
  Tap taps[kMaxTaps];
  uint8_t ksmask[kMaxKBlocks][kMaxTaps];  // 4-bit mask of the 16-channel k-steps to issue
  int32_t nkb, ntaps, nsub, max_dr;
  int32_t mode;
  int32_t n_img, H, W;   // tile-grid space ("A space": output grid, or the low-res grid for kModeUp2)
  int32_t R;             // output rows (of A space) per tile
  int32_t tiles_x, tiles_y, n_chunks, n_tiles;  // n_tiles = n_img*tiles_y*tiles_x*n_chunks
  int32_t n_cta;         // accumulator width N of one CTA tile (<= 64... multiple of 16)
  int32_t acc_stride;    // TMEM columns between accumulators (multiple of 32)
  int32_t a_slots, a_slot_bytes, a_sub_bytes;
  int32_t w_slots, w_slot_bytes, w_tile_bytes;
  int32_t w_resident;    // weights loaded once per CTA
  int32_t desc_mode;     // 0: shifted start; 1: shifted start + base_offset; 2: one box per tap shift
  uint32_t idesc;        // tcgen05 instruction descriptor
  uint32_t a_row_tx;     // bytes one halo row load delivers (all TMA boxes)
  uint32_t w_tx;         // bytes one weight block load delivers
  int32_t* err;          // device int[4]: watchdog diagnostics (tag, block, ...)
  int32_t dbg_flags;     // profiling experiments: 1 skip MMA issue, 2 skip TMA loads, 4 epilogue without math/stores
  int32_t n_in0;         // added to the image coordinate of activation loads (BSVD streaming: ring slot of the frame)
};


// ------------------------------------------------------------------------------------------------
// Row-streaming kernel (conv_stream.cu): 3x3 stride-1 convolutions with the three vertical taps fused
// into the MMA N dimension.  See DESIGN.md section 4.
constexpr int kMaxSKB = 8;          // K blocks (64 input channels each) of one conv
constexpr int kMaxSASlots = 12;     // activation slab ring (one slab = 130 pixels x 64 channels)
constexpr int kMaxAccSlots = 16;    // TMEM accumulator ring (one slot = one output row of 128 pixels)
constexpr int kASlotBytes = 17408;  // 130 * 128 rounded up to the 1024-byte swizzle period

constexpr int kStreamBiasBytes = 1024;  // fp32 bias of every output channel (<= 256 padded channels per conv)

// How a fresh accumulator slot gets its initial value (the bias):
//   NOUT <= 48: the epilogue warp that drained the slot writes the fp32 bias row back with tcgen05.st (the MMA stream is
//               the bound of these variants: no issue slot, no operand traffic spent on it);
//   NOUT == 64: a ones[128x16] x bias_tile[NOUT x 16] MMA issued by the MMA warp (this variant is bound by its epilogue
//               warps -- 2.3 k clk per row against 1.15 k clk of MMAs -- so the 0.5 k clk of tcgen05.st per row cost
//               13 % there while the tensor pipe has the slack).
constexpr bool stream_bias_mma(int nout) { return nout == 64; }
constexpr int kStreamOnesBytes = 128 * 128;  // "ones" operand tile of the bias MMA

constexpr int kStreamEpiWarps = 8;  // two per TMEM lane quarter, alternating output rows
constexpr int kStreamThreads = 32 * (2 + kStreamEpiWarps);
// kOutNV12: chroma hand-over between the two epilogue warps of a lane quarter -- one named barrier per quarter (IDs
// kNv12BarBase .. +3; ID 1 is the set-up barrier) and 2 slots x 4 quarters x 16 pixel pairs of packed 32-bit sums in
// shared memory behind the row records
constexpr int kNv12BarBase = 2;
constexpr int kNv12XchgBytes = 2 * 4 * 16 * 4;
constexpr int kMaskRects = 16;                 // crops per atlas image
constexpr int kMaskStride = 1 + 3 * kMaskRects;  // int32 words per image in StreamParams::mask_hw
constexpr int kStreamSrcWarps = 2;  // frame-format source (StreamParams::src_fmt): decoder warps on top, alternating input rows
constexpr int kStreamThreadsMax = kStreamThreads + 32 * kStreamSrcWarps;

struct StreamParams {
  CUtensorMap tmA[2];   // 5-D (64, W, channel block, H, N), box (64, 130, 1, 1, 1), swizzle 128B
  CUtensorMap tmW;      // 2-D (64, rows), box (64, 3*NOUT): rows = [chunk][kb][kx][2-ky][NOUT], then bias tiles (NOUT == 64)
  CUtensorMap tmB;      // same tensor, box (64, NOUT): the per-chunk bias tile (bias hi/lo in K columns 0/1; NOUT == 64)
  CUtensorMap tmO;      // NHWC output, 4-D (C, W, H, N), box (NOUT, 32, 1, 1), swizzled: TMA store of the fast path
  CUtensorMap tmO2;     // split precision: the same map over the low-half twin of the output tensor
  Epilogue ep;
  // Frame-format source (first layer of the BSVD clip program, north-star part 4): the producer warp decodes the
  // caller's uint8 RGB / NV12 frames itself (/255 or BT.709 limited range, + the constant noise-map channel) straight into
  // the swizzled activation slabs -- no layout kernel, no 16-bit copy of the input read back -- and leaves the decoded
  // rows it owns in src_out (+ src_out_lo) for the DenBlock's residual (out[:, :3] = in[:, :3] - ..., model.py:436-442).
  const uint8_t* src;     // the caller's frames (patched per run)
  int32_t src_fmt;        // 0: activations come through tmA; SS4K_FMT_U8_NHWC (2) or SS4K_FMT_NV12 (3): decoded from src by
                          // kStreamSrcWarps extra warps (launched with kStreamThreadsMax threads)
  int32_t src_fill_ch;    // channel that holds src_fill (3), or -1
  float src_fill;
  uint16_t* src_out;      // [n_total, H, W, 16] 16-bit NHWC, channels 0..7 written
  uint16_t* src_out_lo;   // split precision: low halves, or null
  // Masked canvases / crop atlases (tiled inference, engine.cu::create_tiled_plan): image n of the launch holds up to
  // kMaskRects crops side by side (zero gap columns between them); mask_hw + n * kMaskStride = {count, (x0, w, h) x count}
  // at the plan's input resolution (this conv works at that resolution shifted by mask_shift: > 0 left, < 0 right).
  // Outputs outside every crop are forced to zero, which is what the next conv's zero padding at each crop's own border
  // needs -- crops of different shapes share one image.
  const int32_t* mask_hw;
  int32_t mask_shift;
  int32_t ps2;          // fast store of a PixelShuffle(2) conv (+ skip add): tmO / tmO2 are 5-D (C, b, W, a, N*H) maps over the
                        // shuffled tensor, a chunk is (part of) one sub-pixel phase (a, b); residuals are read at the output pixel
  uint32_t stage_keep;  // fast_store == 0: 1 keeps the (unused) staging region in the shared-memory carve-up (experiments)
  int32_t fast_store;   // 1: plain NHWC output -> registers -> swizzled smem tile -> TMA store;
                        // 2: the same tile stored four times through a 5-D (C, b, W, a, N*H) map: nearest-x2 upsample
                        // 3: split precision (hi + lo twins): two staging tiles per warp, two TMA stores
  const float* bias_f;  // [chunks * NOUT] fp32 bias with alpha folded in: the accumulators' initial value
  int32_t bias_row0;    // first row of the bias tiles inside the weight tensor (NOUT == 64)
  uint8_t a_kb[kMaxSKB];  // source 64-channel block of K block i
  uint8_t a_tm[kMaxSKB];  // which activation tensor map
  uint8_t nks[kMaxSKB];   // 16-channel k-steps to issue (1..4)
  int32_t nkb;
  int32_t n_img, H, W, strips, chunks;
  int32_t total_units;    // chunks * n_img * strips * H output rows of 128 pixels
  int32_t acc_slots, a_slots;
  uint32_t idesc[3];      // instruction descriptors for N = NOUT, 2*NOUT, 3*NOUT
  int32_t* err;
  int32_t dbg_flags;      // profiling experiments (scripts/bench_conv.py, SS4K_DBG_FLAGS): 1 skip MMA issue, 2 skip TMA
                          // loads, 4 epilogue without math / stores, 8 skip band halo rows (WRONG results), 16 full
                          // completion wait on the last output tiles, 64 trace rows stamped by epilogue warp 2
  int32_t n_in0, n_out0;  // added to the image coordinate of TMA loads / stores (BSVD streaming: the frame of image 0)
  // BSVD streams: each tensor is a ring of R frames (R a power of two), and a launch over several frames wraps around it.
  // Image n of the launch lives in slot (n_in0 + n) & ring_in of the input tensor, (n_out0 + n) & ring_out of the output
  // tensor, (n_out0 + n) & ring_res1 / ring_res2 of the residual tensors (mask R - 1; -1 for every other plan: no wrap).
  // The epilogue's pointers (out, out_lo, res1, res2) are at image 0's slot of their tensor.
  int32_t ring_in, ring_out, ring_res1, ring_res2;
  long long* trace;       // debug: per-CTA clock64 stamps [grid][64] (null in production)
  const void* next_w;     // packed weights of the next kernel of the plan (L2 prefetch), or null
  uint32_t next_w_bytes;
  // dead-tensor discard (RRDB dense block): lines of a tensor that no later kernel reads are dropped from L2
  // without write-back (discard.global.L2): 128-byte line l of every pixel with bit l of discard_mask set
  void* discard_ptr;
  uint32_t discard_pitch_bytes, discard_mask;
  int64_t discard_npx;
  // K blocks whose source channels were written at least two kernels ago (dense block: everything but the previous
  // conv's 32 growth channels): their slabs may be loaded before griddepcontrol.wait.  Sound only when this kernel and
  // the two before it fill every SM with one CTA: a CTA of this kernel then runs only after some CTA of the previous
  // kernel has exited, i.e. has itself waited for the kernel before that to complete and flush.
  uint32_t early_kb_mask;
  int32_t l2_in, l2_out;  // L2 eviction priority of the activation loads / output stores: 0 normal, 1 evict_last
                          // (re-read by the next convs of the dense block), 2 evict_first (dead after this conv)
  // Stride-2 convs (BSVD DownBlock, bsvd/model.py:262-263).  The input is read through its pixel-PAIR view
  // (2C channels = [even pixel | odd pixel], W/2 pairs per row): output pixel x needs pair x-1 (odd half, kx = 0) and
  // pair x (even half kx = 1, odd half kx = 2) -> two horizontal shifts with k-step masks instead of three taps.
  // Vertically, input row r feeds output row r/2 (ky = 1) when r is even and output rows (r-1)/2 (ky = 2), (r+1)/2
  // (ky = 0) when r is odd: the weight tile stacks its N blocks as [ky2 | ky0 | ky1] so that both cases are one MMA.
  // H, W are the OUTPUT grid; the activation tensor map has 2 H rows of W pairs.
  // Weight tile group (nkx tiles) read by K block i.  Plain convs: wt[i] = i.  Split precision: the three K blocks of a
  // 64-channel source block are A_hi*W_hi, A_hi*W_lo, A_lo*W_hi -- the first and the third multiply with the SAME weight
  // tiles, which are held once (nwt = 2 groups per source block instead of 3: a third less shared memory for weights,
  // i.e. wider output chunks).
  uint8_t wt[kMaxSKB];
  int32_t nwt;                // distinct weight tile groups of one output chunk
  int32_t stride2;
  int32_t nkx;                // weight tiles (horizontal shifts) per K block: 3, or 2 for stride 2
  uint8_t ksm[kMaxSKB][2];    // stride 2: 4-bit mask of the 16-channel k-steps to issue per (K block, shift)
};

}  // namespace ss4k
