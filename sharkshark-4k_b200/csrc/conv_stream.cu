// Row-streaming tcgen05 / TMEM / TMA implicit-GEMM 3x3 convolution (stride 1, pad 1) for sm_100a.
//
// Replaces torch.nn.Conv2d(k=3) -> cuDNN/TensorRT on the reference's hot path
// (src/upscale/model/realesrgan/factory.py:44-67 SRVGG convs, basicsr RRDBNet convs reached from
//  factory.py:113-125, src/upscale/model/bsvd/model.py:22-53,231-323 BSVD convs).
//
// Formulation (DESIGN.md section 4):
//   * GEMM M = 128 consecutive pixels of one image row (TMEM lanes); K = input channels in 64-channel
//     blocks x 3 horizontal taps; N = 3 vertical taps x NOUT output channels: ONE MMA with N = 3*NOUT
//     adds input row r into the accumulators of output rows r-1, r, r+1, which sit side by side in a
//     ring of TMEM accumulator slots.  Versus one MMA per tap this reads the activation operand from
//     shared memory 3x less often (the bound for small Cout) and issues 3x fewer instructions.
//   * the three horizontal taps are the same 130-pixel halo slab addressed with a 0/1/2-row shifted
//     start address (swizzle-128B K-major descriptors), so no im2col and no re-read of activations.
//   * a CTA owns a contiguous run of output rows of one 128-pixel column strip and STREAMS input rows
//     through a shared-memory ring: every input row is loaded once (2 halo rows per band), the MMA
//     stream never drains between rows, and the epilogue warps retire output row y as soon as input
//     row y+1 has been accumulated.  Rows are split evenly over the persistent grid (one CTA per SM).
//   * all weights of the conv (every K block and tap) stay resident in shared memory.
//   * accumulator slots start from the bias, so every MMA accumulates: the 16/32/48-wide variants have the epilogue
//     warp that drained a slot (tcgen05.ld) write the fp32 bias row back (tcgen05.st) -- no issue slot, no operand
//     traffic; the 64-wide variant, whose tensor pipe has the slack, uses a ones x bias-tile MMA (conv_params.h,
//     stream_bias_mma).
//   * warp 0 = TMA producer and row planner, warp 1 = MMA issuer, warps 2..9 = epilogue, two warps per TMEM lane
//     quarter taking alternate output rows: TMEM -> registers -> activation / scaled residual adds ->
//     16-bit pack -> swizzled shared-memory tile -> TMA store (plain NHWC outputs).  The epilogue warps share the
//     SM's four schedulers with the MMA-issuing warp, so their arithmetic is specialised per shape (`emode`: 2-4
//     instructions per value instead of ~20 for the general form); uint8 RGB rows, PixelShuffle(4) into half NCHW
//     and BSVD's ReLU6 / PixelShuffle(2) + skip / temporal-shift scatter stores have lean paths of their own, the
//     rest (NCHW float, hi+lo split stores, ...) goes through epilogue_chunk.
//   * memory system: L2 eviction-priority hints on the TMA loads / stores and discard of dead slab lines (dense
//     block, DESIGN.md section 4.4); K blocks that only read channels of older kernels are requested before the
//     dependency wait (early_kb_mask); the next kernel's weights are prefetched into L2.
//   * NOTE for maintainers: a 64-bit integer division or any out-of-line call in this kernel makes ptxas give up
//     the uniform registers of the MMA issue loop (R2UR count 69 -> 270, -30 %): check
//     `cuobjdump -sass libss4k.so | grep -c R2UR` for the <32> variant after every change.
//   * row records: the accumulator-ring bookkeeping of every input row (which slots it touches first / completes,
//     where the ring wraps, descriptors, chunk switches) is computed by the producer warp and travels with the
//     row's first activation slab as a 32-byte record; the issuing warp reads the NEXT row's record and waits for
//     its fresh (bias-initialised) accumulator slot in the middle of the current row's last burst, so the tensor
//     pipe's queue (about 6 instructions, scripts/mma_issue_probe.cu) never drains at a row boundary.
//   * fp16 hi/lo split operands (BSVD precision mode): three K blocks per 64 source channels
//     (A_hi*W_hi, A_hi*W_lo, A_lo*W_hi), the low halves through a second activation tensor map.
//   * measured bound (DESIGN.md section 4.1): an M=128, N=96, K=16 MMA costs 56 clk of shared-memory port time for
//     48 clk of math; with the slab written by TMA and the epilogue's staging tile the port carries about 117 KB
//     per row of a 64->32 conv, which sets the row period the kernel runs at.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv_common.cuh"
#include "conv_params.h"

namespace ss4k {

namespace {

__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(pred));
  return pred;
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

constexpr uint64_t kSdescHi = (static_cast<uint64_t>(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
__device__ __forceinline__ uint64_t sdesc(uint32_t saddr) {
  return kSdescHi | static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
}

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5}], [%1], %6;"
               :
               : "l"(reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3, int c4, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5, %6}], [%1], %7;"
               :
               : "l"(reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(pol)
               : "memory");
}
// programmatic dependent launch: let the next kernel of the stream start its prologue early / wait for the
// previous kernel's results before touching them
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// row record flags (word 5; bits 0..1 = accumulator blocks after the ring wrap)
constexpr uint32_t kRecLast = 4u, kRecNewChunk = 8u, kRecFreeW = 16u;
constexpr uint32_t kRecWords = 8u;

struct Band {
  int chunk, n, strip, yb, ye;
};
// units are output rows in (chunk, n, strip, y) order; a band is a run of rows inside one strip
__device__ __forceinline__ bool next_band(const StreamParams& P, int& u, int u1, Band& b) {
  if (u >= u1) return false;
  int t = u;
  const int y = t % P.H;
  t /= P.H;
  b.strip = t % P.strips;
  t /= P.strips;
  b.n = t % P.n_img;
  b.chunk = t / P.n_img;
  b.yb = y;
  const int rem = u1 - u;
  b.ye = rem < P.H - y ? y + rem : P.H;
  u += b.ye - b.yb;
  return true;
}

// Image n of the launch in the ring buffers of a BSVD stream (StreamParams::ring_*): the output / residual image indices
// relative to the epilogue's base pointers, and the distances to frames n-1 / n+1 in the output ring (they wrap with it).
// Every other plan has masks of -1: image n, one frame either side.
__device__ __forceinline__ int ring_n(const StreamParams& P, int n, int mask) { return ((P.n_out0 + n) & mask) - (P.n_out0 & mask); }
__device__ __forceinline__ ImgAt ring_img(const StreamParams& P, int n) {
  const int f = P.n_out0 + n;
  const int so = f & P.ring_out;
  ImgAt I;
  I.out = so - (P.n_out0 & P.ring_out);
  I.res1 = ring_n(P, n, P.ring_res1);
  I.res2 = ring_n(P, n, P.ring_res2);
  I.t = P.ep.t0 + n;
  I.prev = so - ((f - 1) & P.ring_out);
  I.next = ((f + 1) & P.ring_out) - so;
  return I;
}

}  // namespace

static_assert(kMaxSASlots <= 16 && kMaxAccSlots <= 16, "barrier set-up assigns one lane per ring slot");

// ---- frame-format source of the first layer (StreamParams::src): same arithmetic as prep_kernel (elementwise.cu).
// A lane owns four consecutive interior pixels of the 130-pixel halo row (slab pixels 1 + 4 lane + i, aligned 32-bit
// loads: W % 4 == 0) and lanes 0 / 31 the left / right halo pixel on top.
struct SrcPix { uint32_t hi[2], lo[2]; };   // channels 0..3 as 16-bit pairs (value = hi + lo)
struct SrcRow { uint32_t w[3], extra; };    // raw bytes: NV12 {Y x4, UV x2 pairs, -}, RGB {12 bytes}; extra: the halo pixel's three
                                            // bytes (Y | U << 8 | V << 16 or R | G << 8 | B << 16) | bit 24: it exists | bit 25: the interior group exists
constexpr uint32_t kSrcNone = 0xFFFFFFFFu;  // pixel outside the frame (zero padding)
__device__ __forceinline__ SrcRow src_load_row(const StreamParams& P, int n, int r, int x4, int xe) {
  SrcRow o;
  o.w[0] = o.w[1] = o.w[2] = 0u;
  o.extra = 0u;
  const bool in4 = x4 < P.W, ine = xe >= 0 && xe < P.W;
  if (P.src_fmt == 3) {
    const uint8_t* frame = P.src + static_cast<size_t>(n) * (static_cast<size_t>(P.H) * P.W * 3 / 2);
    const uint8_t* yrow = frame + static_cast<size_t>(r) * P.W;
    const uint8_t* uvrow = frame + static_cast<size_t>(P.H) * P.W + static_cast<size_t>(r >> 1) * P.W;
    if (in4) {
      o.w[0] = __ldg(reinterpret_cast<const uint32_t*>(yrow + x4));
      o.w[1] = __ldg(reinterpret_cast<const uint32_t*>(uvrow + x4));
    }
    if (ine)
      o.extra = static_cast<uint32_t>(__ldg(yrow + xe)) | (static_cast<uint32_t>(__ldg(reinterpret_cast<const uint16_t*>(uvrow + (xe & ~1)))) << 8);
  } else {
    const uint8_t* row = P.src + (static_cast<size_t>(n) * P.H + r) * P.W * 3;
    if (in4) {
      const uint32_t* q = reinterpret_cast<const uint32_t*>(row + static_cast<size_t>(x4) * 3);
      o.w[0] = __ldg(q); o.w[1] = __ldg(q + 1); o.w[2] = __ldg(q + 2);
    }
    if (ine) {
      const uint8_t* px = row + static_cast<size_t>(xe) * 3;
      o.extra = static_cast<uint32_t>(__ldg(px)) | (static_cast<uint32_t>(__ldg(px + 1)) << 8) | (static_cast<uint32_t>(__ldg(px + 2)) << 16);
    }
  }
  o.extra |= (ine ? 1u << 24 : 0u) | (in4 ? 1u << 25 : 0u);
  return o;
}
__device__ __forceinline__ SrcPix src_decode(const StreamParams& P, uint32_t raw) {   // raw: three bytes, or kSrcNone
  SrcPix o;
  o.hi[0] = o.hi[1] = o.lo[0] = o.lo[1] = 0u;
  if (raw == kSrcNone) return o;
  float v[4];
  const float b0 = static_cast<float>(raw & 0xFFu), b1 = static_cast<float>((raw >> 8) & 0xFFu), b2 = static_cast<float>((raw >> 16) & 0xFFu);
  if (P.src_fmt == 3) {  // BT.709 limited range, nearest chroma
    const float yy = (b0 - 16.f) * (1.f / 219.f);
    const float cb = (b1 - 128.f) * (1.f / 224.f);
    const float cr = (b2 - 128.f) * (1.f / 224.f);
    v[0] = fminf(fmaxf(yy + 1.5748f * cr, 0.f), 1.f);
    v[1] = fminf(fmaxf(yy - 0.187324f * cb - 0.468124f * cr, 0.f), 1.f);
    v[2] = fminf(fmaxf(yy + 1.8556f * cb, 0.f), 1.f);
  } else {
    v[0] = b0 / 255.0f; v[1] = b1 / 255.0f; v[2] = b2 / 255.0f;
  }
  v[3] = P.src_fill_ch == 3 ? P.src_fill : 0.f;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn(v[2 * i] - back.x, v[2 * i + 1] - back.y);
    o.hi[i] = *reinterpret_cast<const uint32_t*>(&h);
    o.lo[i] = *reinterpret_cast<const uint32_t*>(&l);
  }
  return o;
}
// the three source bytes of interior pixel i (0..3) of a lane's row / of its halo pixel, or kSrcNone
__device__ __forceinline__ uint32_t src_px(const StreamParams& P, const SrcRow& R, int i) {
  if (!(R.extra & (1u << 25))) return kSrcNone;
  if (P.src_fmt == 3) return ((R.w[0] >> (8 * i)) & 0xFFu) | (((R.w[1] >> (16 * (i >> 1))) & 0xFFFFu) << 8);
  const uint64_t lo = (static_cast<uint64_t>(R.w[1]) << 32) | R.w[0];
  const uint64_t hi = (static_cast<uint64_t>(R.w[2]) << 32) | R.w[1];
  return i < 2 ? static_cast<uint32_t>(lo >> (24 * i)) & 0xFFFFFFu : static_cast<uint32_t>(hi >> (24 * i - 32)) & 0xFFFFFFu;
}
__device__ __forceinline__ uint32_t src_px_extra(const SrcRow& R) { return (R.extra & (1u << 24)) ? (R.extra & 0xFFFFFFu) : kSrcNone; }

// L2 prefetch of the source bytes of input row r of a strip (lane l < 3 takes one 128-byte line): the decoder warps'
// register prefetch (one of their rows ahead) then hits L2 instead of paying a DRAM round trip per row
__device__ __forceinline__ void src_prefetch_row(const StreamParams& P, int n, int r, int xs, int l) {
  const uint8_t* p;
  if (P.src_fmt == 3) {
    if (l >= 2) return;
    const uint8_t* frame = P.src + static_cast<size_t>(n) * (static_cast<size_t>(P.H) * P.W * 3 / 2);
    p = l == 0 ? frame + static_cast<size_t>(r) * P.W + xs : frame + static_cast<size_t>(P.H) * P.W + static_cast<size_t>(r >> 1) * P.W + xs;
  } else {
    if (l >= 3) return;
    p = P.src + ((static_cast<size_t>(n) * P.H + r) * P.W + xs) * 3 + 128 * l;
  }
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

template <int NOUT>
__global__ void __launch_bounds__(kStreamThreadsMax, 1)
conv3x3_stream_kernel(const __grid_constant__ StreamParams P) {
  extern __shared__ uint8_t smem_raw[];
  constexpr uint32_t kWTile = 3u * NOUT * 128u;      // one (K block, horizontal tap) weight tile
  constexpr uint32_t kStageWarp = 32u * NOUT * 2u;   // one epilogue warp's 32-pixel output tile
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = smem_base;
  // after the weights: fp32 bias of every chunk (tcgen05.st initialisation), or bias tile + ones tile (bias MMA)
  constexpr bool kBiasMMA = stream_bias_mma(NOUT);
  constexpr uint32_t kBiasTile = NOUT * 128u;
  const uint32_t bias_base = w_base + static_cast<uint32_t>(P.nwt * P.nkx) * kWTile;
  const uint32_t ones_base = bias_base + kBiasTile;
  const uint32_t a_base = kBiasMMA ? ones_base + kStreamOnesBytes : bias_base + kStreamBiasBytes;
  const uint32_t stage_base = a_base + static_cast<uint32_t>(P.a_slots) * kASlotBytes;
  // (split-precision fast store: a second tile per warp for the low halves)
  const uint32_t stage_stride = P.fast_store == 0 ? P.stage_keep * ((kStageWarp + 1023u) & ~1023u)
                                                  : (((P.fast_store == 3 ? 2u * kStageWarp : kStageWarp) + 1023u) & ~1023u);
  const uint32_t bar_base = stage_base + kStreamEpiWarps * stage_stride;
  const uint32_t a_full = bar_base;
  const uint32_t a_empty = a_full + 8 * kMaxSASlots;
  const uint32_t acc_full = a_empty + 8 * kMaxSASlots;
  const uint32_t acc_empty = acc_full + 8 * kMaxAccSlots;
  const uint32_t w_full = acc_empty + 8 * kMaxAccSlots;
  const uint32_t w_empty = w_full + 8;
  const uint32_t tmem_slot = w_empty + 8;
  const uint32_t rec_base = tmem_slot + 32;  // row records, one per activation slab slot (kRecWords x 4 bytes each)
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);  // warp-uniform for ptxas
  const int lane = threadIdx.x & 31;
  long long* const trace = P.trace != nullptr ? P.trace + blockIdx.x * 128 : nullptr;
#define SS4K_TRACE(i) do { if (trace != nullptr && lane == 0) trace[i] = clock64(); } while (0)
  if (warp == 0) SS4K_TRACE(0);

  pdl_launch_dependents();
  {
    // touch every 64-byte line of the parameter block at once: the first use of each field otherwise misses in the
    // constant cache one after the other along the set-up path
    const uint64_t* pw = reinterpret_cast<const uint64_t*>(&P);
    uint64_t acc = 0;
#pragma unroll
    for (int i = 0; i < static_cast<int>(sizeof(StreamParams) / 64); ++i) acc ^= pw[i * 8];
    asm volatile("" ::"l"(acc));
  }
  // NV12 store: rows are split in pairs, so that both rows of a chroma row pair belong to one CTA and (H even) every
  // band starts on an even row: the row counter's parity is the row's parity, row 2j goes to the parity-0 warp and row
  // 2j+1 to the parity-1 warp of the same lane quarter
  const int pair_sh = (NOUT == 16 && P.ep.out_mode == kOutNV12) ? 1 : 0;
  const int u0 = static_cast<int>(static_cast<int64_t>(blockIdx.x) * (P.total_units >> pair_sh) / gridDim.x) << pair_sh;
  const int u1 = static_cast<int>(static_cast<int64_t>(blockIdx.x + 1) * (P.total_units >> pair_sh) / gridDim.x) << pair_sh;
  int early_chunk = -1;  // weights requested in the prologue (producer warp)
  if (warp == 0) {
    // barrier set-up spread over the warp's lanes (58 dependent shared-memory operations from one lane were a
    // visible part of the per-launch fixed cost)
    if (lane == 0) {
      prefetch_tmap(&P.tmA[0]);
      prefetch_tmap(&P.tmW);
      if (kBiasMMA) prefetch_tmap(&P.tmB);
      if (P.fast_store) prefetch_tmap(&P.tmO);
      mbar_init(w_full, 1);
      mbar_init(w_empty, 1);
    }
    if (lane < kMaxSASlots) {
      mbar_init(a_full + 8 * lane, P.src_fmt != 0 ? 2 : 1);   // frame-format source: the row record (this warp) + the decoded slab
      mbar_init(a_empty + 8 * lane, 1);
    }
    if (lane >= 16 && lane < 16 + kMaxAccSlots) {
      mbar_init(acc_full + 8 * (lane - 16), 1);
      mbar_init(acc_empty + 8 * (lane - 16), 4);  // one arrive per epilogue warp of the row's parity group
    }
    fence_barrier_init();
    __syncwarp();
    // the first chunk's weights are constants of the launch: request them before the rest of the set-up
    // (TMEM allocation, bias copy, block barrier) so that their latency overlaps it
    if (u0 < u1) {
      int uu = u0;
      Band fb;
      next_band(P, uu, u1, fb);
      early_chunk = fb.chunk;
      if (elect_one()) {
        const int ntile = P.nwt * P.nkx;
        mbar_expect_tx(w_full, static_cast<uint32_t>(ntile) * kWTile + (kBiasMMA ? kBiasTile : 0u));
        for (int t = 0; t < ntile; ++t)
          tma_load_2d(w_base + t * kWTile, &P.tmW, w_full, 0, (fb.chunk * ntile + t) * 3 * NOUT);
        if (kBiasMMA) tma_load_2d(bias_base, &P.tmB, w_full, 0, P.bias_row0 + fb.chunk * NOUT);
      }
      __syncwarp();
    }
    SS4K_TRACE(9);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    SS4K_TRACE(10);
  }
  {
    // fp32 bias of every output channel (alpha already folded in): the epilogue warps write it into the accumulator
    // slots they own.  A constant of the launch, so it is read before the dependency wait.
    if (kBiasMMA) {
      // "ones" operand of the accumulator-init MMA: 128 rows x 64 channels, swizzle-128B K-major, value 1 in K
      // columns 0 and 1 (they meet the hi / lo halves of the bias in the bias tile), 0 elsewhere
      const uint32_t one2 = P.ep.is_bf16 ? 0x3F803F80u : 0x3C003C00u;
      if (warp != 0 && warp < 2 + kStreamEpiWarps)
        for (uint32_t ci = threadIdx.x - 32; ci < 1024u; ci += kStreamThreads - 32) {
          const uint32_t r = ci >> 3, pc = ci & 7u;
          sts128(ones_base + ci * 16u, pc == (r & 7u) ? one2 : 0u, 0u, 0u, 0u);
        }
      fence_proxy_async();
    } else {
      float* sb = reinterpret_cast<float*>(smem_gen + (bias_base - smem_base));
      const int nb = P.chunks * NOUT;
      if (warp != 0 && warp < 2 + kStreamEpiWarps)
        for (int i = threadIdx.x - 32; i < nb; i += kStreamThreads - 32) sb[i] = __ldg(P.bias_f + i);
    }
    if (warp == 2) SS4K_TRACE(11);
  }
  // Set-up barrier: the producer warp only ARRIVES (its barrier initialisation becomes visible to the others) and goes
  // straight on to its loads -- it needs neither the TMEM allocation nor the bias copy, and its first activation
  // load is the head of the per-launch critical path.
  if (warp == 0) {
    asm volatile("bar.arrive 1, %0;" ::"r"(blockDim.x) : "memory");
  } else {
    tcgen05_before_sync();
    asm volatile("bar.sync 1, %0;" ::"r"(blockDim.x) : "memory");
    tcgen05_after_sync();
    // this CTA owns all 512 TMEM columns (one CTA per SM), so the allocation starts at column 0 / lane 0;
    // using the constant keeps TMEM addresses in uniform registers
    if (*tmem_slot_ptr != 0u) __trap();
  }
  constexpr uint32_t tmem_base = 0u;
  if (warp == 1) SS4K_TRACE(1);

  const int S = P.acc_slots;

  if (warp == 0) {
    // ======================================================= TMA producer + row planner
    // Besides the loads, this warp does the per-row bookkeeping of the MMA stream (accumulator ring positions,
    // which slots an input row touches first / completes, where the ring wraps) and hands it to the MMA
    // warp as a small record that travels with the row's first activation slab: the issuing warp is the
    // critical resource of the kernel (one thread feeds the tensor pipe), this one has time to spare.
    uint32_t as = 0, aph = 0, wph = 0;
    int loaded_chunk = -1;
    int u = u0;
    const uint64_t pol_in = l2_policy(P.l2_in);
    Band b, nb;
    bool dep_ready = false;
    int prow = 0;        // traced rows
    int sL = 0, kL = 0;  // accumulator ring position (slot, wrap count) of output row y_lo
    bool has = next_band(P, u, u1, b);
    const bool from_src = P.src_fmt != 0;   // the slabs are filled by the decoder warps; this warp sends the row records
    while (has) {
      const bool has_next = next_band(P, u, u1, nb);
      const bool new_chunk = b.chunk != loaded_chunk;
      if (new_chunk) {
        mbar_wait_u(w_empty, wph ^ 1);
        if (b.chunk == early_chunk) {
          early_chunk = -1;  // already requested in the prologue
        } else if (elect_one()) {
          const int ntile = P.nwt * P.nkx;
          mbar_expect_tx(w_full, static_cast<uint32_t>(ntile) * kWTile + (kBiasMMA ? kBiasTile : 0u));
          for (int t = 0; t < ntile; ++t)
            tma_load_2d(w_base + t * kWTile, &P.tmW, w_full, 0, (b.chunk * ntile + t) * 3 * NOUT);
          if (kBiasMMA) tma_load_2d(bias_base, &P.tmB, w_full, 0, P.bias_row0 + b.chunk * NOUT);
        }
        __syncwarp();
        wph ^= 1;
        loaded_chunk = b.chunk;
      }
      // (weights are constants; the activations belong to earlier kernels of the stream: the dependency wait sits in
      //  front of the first load that may touch the PREVIOUS kernel's output, see StreamParams::early_kb_mask)
      if (!dep_ready && P.early_kb_mask == 0u) {
        SS4K_TRACE(12);
        pdl_wait();
        dep_ready = true;
        SS4K_TRACE(13);
      }
      // dbg_flags & 8: skip the band's halo rows (WRONG results at band boundaries; measures what they cost)
      const bool s2 = P.stride2 != 0;
      int r0, r1;
      if (s2) {  // output rows [yb, ye) read input rows [2 yb - 1, 2 ye - 1]
        r0 = b.yb > 0 ? 2 * b.yb - 1 : 0;
        r1 = 2 * b.ye - 1;
      } else {
        r0 = (b.yb > 0 && !(P.dbg_flags & 8)) ? b.yb - 1 : b.yb;
        r1 = (b.ye < P.H && !(P.dbg_flags & 8)) ? b.ye : b.ye - 1;
      }
      const int x0 = b.strip * kTileW - 1;
      int y_lo = b.yb;
      for (int r = r0; r <= r1; ++r) {
        const bool ptr8 = trace != nullptr && lane == 0 && prow == 8;
        if (trace != nullptr && lane == 0 && prow < 16) trace[64 + prow++] = clock64();
        // ---- the row's record: output rows [y_lo, y_hi] receive this input row, the first through weight block b_lo
        int y_first, y_hi, b_lo, f_lo;
        bool done_lo;  // this input row completes output row y_lo
        if (s2) {
          if (r & 1) {
            const int ya = (r - 1) >> 1;  // ky = 2 for row ya (block 0), ky = 0 for row ya + 1 (block 1)
            y_first = ya > b.yb ? ya : b.yb;
            y_hi = ya + 1 < b.ye - 1 ? ya + 1 : b.ye - 1;
            b_lo = y_first - ya;
            f_lo = ya + 1;
            done_lo = ya >= b.yb;
          } else {                        // ky = 1 (block 2)
            y_first = y_hi = r >> 1;
            b_lo = 2;
            f_lo = y_hi + 1;
            done_lo = false;
          }
        } else {
          y_first = r - 1 > b.yb ? r - 1 : b.yb;
          y_hi = r + 1 < b.ye - 1 ? r + 1 : b.ye - 1;
          b_lo = y_first - (r - 1);  // weight row block (block = 2 - ky) of output row y_lo
          f_lo = r + 1;
          done_lo = r - 1 >= b.yb;
        }
        if (y_first != y_lo) {
          y_lo = y_first;
          if (++sL == S) { sL = 0; ++kL; }
        }
        if (r == r0) f_lo = y_lo;
        const int nblk = y_hi - y_lo + 1;
        const int nA = sL + nblk <= S ? nblk : S - sL;  // the MMAs split where the ring wraps
        const int nB = nblk - nA;
        uint32_t fresh = 0;  // up to 3 x {bit 7 valid, bit 6 parity of the slot's use count, bits 0..4 slot}
        {
          int sh = 0;
          for (int y = f_lo; y <= y_hi; ++y, sh += 8) {
            int s2_ = sL + (y - y_lo), k2 = kL;
            if (s2_ >= S) { s2_ -= S; ++k2; }
            fresh |= (0x80u | ((k2 & 1) ? 0x40u : 0u) | static_cast<uint32_t>(s2_)) << sh;
          }
        }
        uint32_t c0 = 0xFFu, c1 = 0xFFu;  // accumulator slots completed by this input row
        if (done_lo) c0 = static_cast<uint32_t>(sL);
        if (!s2 && r == r1 && r <= b.ye - 1) {  // image bottom: row H-1 has no row below it
          int s2_ = sL + (r - y_lo);
          if (s2_ >= S) s2_ -= S;
          c1 = static_cast<uint32_t>(s2_);
        }
        const uint32_t flags = static_cast<uint32_t>(nB) | ((r == r1 && !has_next) ? kRecLast : 0u) |
                               ((r == r0 && new_chunk) ? kRecNewChunk : 0u) |
                               ((r == r1 && has_next && nb.chunk != b.chunk) ? kRecFreeW : 0u);
        if (ptr8) trace[112] = clock64();
        for (int kb = 0; kb < P.nkb; ++kb) {
          if (!dep_ready && !((P.early_kb_mask >> kb) & 1u)) {
            SS4K_TRACE(12);
            pdl_wait();
            dep_ready = true;
            SS4K_TRACE(13);
          }
          mbar_wait_u(a_empty + 8 * as, aph ^ 1);
          if (ptr8) trace[113] = clock64();
          if (from_src) {
            if (lane == 0) {
              if (kb == 0) {
                const uint32_t ra = rec_base + as * (kRecWords * 4u);
                sts128(ra, static_cast<uint32_t>(sL * NOUT), P.idesc[nA - 1], P.idesc[nB > 0 ? nB - 1 : 0],
                       static_cast<uint32_t>(b_lo * NOUT * 128) >> 4);
                sts128(ra + 16, static_cast<uint32_t>((b_lo + nA) * NOUT * 128) >> 4, flags, c0 | (c1 << 8), fresh);
              }
              mbar_arrive(a_full + 8 * as);
            }
          } else if (elect_one()) {
            if (kb == 0) {
              const uint32_t ra = rec_base + as * (kRecWords * 4u);
              sts128(ra, static_cast<uint32_t>(sL * NOUT), P.idesc[nA - 1], P.idesc[nB > 0 ? nB - 1 : 0],
                     static_cast<uint32_t>(b_lo * NOUT * 128) >> 4);
              sts128(ra + 16, static_cast<uint32_t>((b_lo + nA) * NOUT * 128) >> 4, flags, c0 | (c1 << 8), fresh);
            }
            if (P.dbg_flags & 2) {
              mbar_arrive(a_full + 8 * as);
            } else {
              mbar_expect_tx(a_full + 8 * as, kBoxW * kRowBytes);
              tma_load_5d_hint(a_base + as * kASlotBytes, &P.tmA[P.a_tm[kb]], a_full + 8 * as, 0, x0, P.a_kb[kb], r, (b.n + P.n_in0) & P.ring_in, pol_in);
            }
          }
          if (ptr8) trace[114] = clock64();
          __syncwarp();
          if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
          if (ptr8) trace[115] = clock64();
        }
      }
      // ring position of the next band's first output row
      sL += b.ye - y_lo;
      if (sL >= S) { sL -= S; ++kL; }
      b = nb;
      has = has_next;
    }
    // all loads of this CTA are in flight: pull this CTA's share of the NEXT kernel's weights into L2 (they were
    // evicted by a frame's worth of activations since their last use; an HBM miss would sit on its prologue)
    if (P.next_w != nullptr && lane == 0) {
      const uint32_t per = ((P.next_w_bytes + gridDim.x - 1) / gridDim.x + 15u) & ~15u;
      const uint32_t off = blockIdx.x * per;
      if (off < P.next_w_bytes) {
        const uint32_t sz = P.next_w_bytes - off < per ? ((P.next_w_bytes - off) & ~15u) : per;
        if (sz > 0)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const uint8_t*>(P.next_w) + off), "r"(sz) : "memory");
      }
    }
  } else if (warp == 1) {
    // ======================================================= MMA issuer
    // The whole warp runs this loop convergently (waits are asm-internal loops, record words are broadcast
    // with shuffles) so that ptxas keeps every descriptor in uniform registers; one elected lane issues the
    // tcgen05 instructions.  One thread feeds the tensor pipe and the pipe queues almost nothing, so every
    // instruction this warp executes between two MMAs is dead time for the pipe: the row bookkeeping comes
    // precomputed from the producer warp (row records), and the next row's record and its fresh accumulator slots
    // (wait for the epilogue's drain + bias re-initialisation) are handled in the middle of the current row's last burst.
    uint32_t as = 0, aph = 0, wph = 0;
    const int nkb = P.nkb;
    const bool do_mma = !(P.dbg_flags & 1);
    const uint32_t n_aslots = static_cast<uint32_t>(P.a_slots);

    uint32_t rc[kRecWords];
    // waits for the first slab of a row, reads its record and prepares its fresh accumulator slots
    auto fetch = [&](uint32_t slot, uint32_t ph) {
      mbar_wait_u(a_full + 8 * slot, ph);
      uint32_t v0, v1, v2, v3, v4, v5, v6, v7;
      const uint32_t ra = rec_base + slot * (kRecWords * 4u);
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3) : "r"(ra) : "memory");
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v4), "=r"(v5), "=r"(v6), "=r"(v7) : "r"(ra + 16) : "memory");
      rc[0] = __shfl_sync(0xffffffffu, v0, 0); rc[1] = __shfl_sync(0xffffffffu, v1, 0);
      rc[2] = __shfl_sync(0xffffffffu, v2, 0); rc[3] = __shfl_sync(0xffffffffu, v3, 0);
      rc[4] = __shfl_sync(0xffffffffu, v4, 0); rc[5] = __shfl_sync(0xffffffffu, v5, 0);
      rc[6] = __shfl_sync(0xffffffffu, v6, 0); rc[7] = __shfl_sync(0xffffffffu, v7, 0);
    };
    auto prepare = [&]() {  // rc = record of the row about to be issued
      if (rc[5] & kRecNewChunk) {
        mbar_wait_u(w_full, wph);
        wph ^= 1;
        if (trace != nullptr && lane == 0 && trace[2] == 0) trace[2] = clock64();
      }
      tcgen05_after_sync();
      uint32_t f = rc[7];
#pragma unroll
      for (int j = 0; j < 3; ++j, f >>= 8) {
        if (f & 0x80u) {  // fresh slot: drained (and, NOUT <= 48, re-initialised with the bias) by the epilogue warps
          mbar_wait_u(acc_empty + 8 * (f & 0x1Fu), (f >> 6) & 1u);
          tcgen05_after_sync();
          if (kBiasMMA && do_mma) umma_f16_elect(tmem_base + (f & 0x1Fu) * NOUT, sdesc(ones_base), sdesc(bias_base), P.idesc[0], 0u);
        }
      }
    };

    if (u0 < u1) {
      fetch(0, 0);
      prepare();
      SS4K_TRACE(3);
      bool last = false;
      int rowcnt = 0;
      while (!last) {
        // this row's plan in uniform registers
        const uint32_t colA = tmem_base + rc[0], idA = rc[1], idB = rc[2], woffA = rc[3], woffB = rc[4];
        const uint32_t flags = rc[5], cc = rc[6];
        const bool wrap = (flags & 3u) != 0;
        last = (flags & kRecLast) != 0;
        // (a row that frees the weights cannot look ahead: the next row's weights load after its last MMA)
        const bool overlap = !last && !(flags & kRecFreeW);
        const bool trow = trace != nullptr && lane == 0 && rowcnt < 8;
        long long* const trw = trace + 16 + 6 * rowcnt;
        if (trow) trw[0] = clock64();
        for (int kb = 0; kb < nkb; ++kb) {
          if (kb > 0) {
            mbar_wait_u(a_full + 8 * as, aph);
            tcgen05_after_sync();
          }
          // descriptor low words (address >> 4): per-MMA offsets are compile-time constants
          const uint32_t a_lo = (a_base + as * kASlotBytes) >> 4;
          const uint32_t w_lo = (w_base + static_cast<uint32_t>(P.wt[kb] * P.nkx) * kWTile) >> 4;
          const uint32_t wA_lo = w_lo + woffA, wB_lo = w_lo + woffB;
          const int nks = P.nks[kb];
          const uint32_t as_cur = as;
          if (++as == n_aslots) { as = 0; aph ^= 1; }
#define SS4K_MMA(KX, KS)                                                                                                   \
          {                                                                                                                \
            umma_f16_lo(colA, a_lo + ((KX) * kRowBytes + (KS) * 32) / 16, wA_lo + ((KX) * kWTile + (KS) * 32) / 16, idA, 1u); \
            if (wrap) umma_f16_lo(tmem_base, a_lo + ((KX) * kRowBytes + (KS) * 32) / 16, wB_lo + ((KX) * kWTile + (KS) * 32) / 16, idB, 1u); \
          }
          if (P.stride2) {
            // pixel-pair view: shift 0 = pair x-1 (odd half only), shift 1 = pair x; k-steps from the per-shift masks
            const uint32_t m0 = P.ksm[kb][0], m1 = P.ksm[kb][1];
            if (do_mma) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                if ((m0 >> ks) & 1u) SS4K_MMA(0, ks)
            }
            if (kb == nkb - 1 && overlap) {
              fetch(as, aph);
              prepare();
            }
            if (do_mma) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                if ((m1 >> ks) & 1u) SS4K_MMA(1, ks)
            }
          } else {
          if (do_mma) {
            if (nks == 4) {
              SS4K_MMA(0, 0) SS4K_MMA(0, 1) SS4K_MMA(0, 2) SS4K_MMA(0, 3)
              SS4K_MMA(1, 0) SS4K_MMA(1, 1) SS4K_MMA(1, 2) SS4K_MMA(1, 3)
            } else {
#pragma unroll
              for (int kx = 0; kx < 2; ++kx) {
#pragma unroll
                for (int ks = 0; ks < 3; ++ks)
                  if (ks < nks) SS4K_MMA(kx, ks)
              }
            }
          }
          if (trow && kb == nkb - 1) trw[1] = clock64();
          if (kb == nkb - 1 && overlap) {  // next row: first slab, record, fresh accumulator slots
            fetch(as, aph);
            if (trow) trw[2] = clock64();
            prepare();
          }
          if (trow && kb == nkb - 1) trw[3] = clock64();
          if (do_mma) {
            if (nks == 4) {
              SS4K_MMA(2, 0) SS4K_MMA(2, 1) SS4K_MMA(2, 2) SS4K_MMA(2, 3)
            } else {
#pragma unroll
              for (int ks = 0; ks < 3; ++ks)
                if (ks < nks) SS4K_MMA(2, ks)
            }
          }
          }
#undef SS4K_MMA
          umma_commit_elect(a_empty + 8 * as_cur);  // slab reusable once these MMAs have read it
        }
        if (trow) trw[4] = clock64();
        // ---- output rows completed by this input row
        if ((cc & 0xFFu) != 0xFFu) umma_commit_elect(acc_full + 8 * (cc & 0xFFu));
        if (((cc >> 8) & 0xFFu) != 0xFFu) umma_commit_elect(acc_full + 8 * ((cc >> 8) & 0xFFu));
        if (flags & kRecFreeW) umma_commit_elect(w_empty);  // weights may be replaced
        if (!last && !overlap) {
          fetch(as, aph);
          prepare();
        }
        if (trow) trw[5] = clock64();
        ++rowcnt;
      }
    }
    SS4K_TRACE(4);
  } else if (warp >= 2 + kStreamEpiWarps) {
    // ======================================================= frame decoders (frame-format source only)
    // Warp d of kStreamSrcWarps takes every kStreamSrcWarps-th input row of the producer's sequence: loads the row's
    // bytes (the next one of its rows is in flight meanwhile), converts, writes the row's activation slabs -- the same
    // swizzled layout a TMA box load produces, one per K block (split precision: high, high, low halves) -- and the
    // 16-bit copy for the DenBlock's residual.
    const int dw = warp - (2 + kStreamEpiWarps);
    const int src_xe_off = lane == 0 ? -1 : (lane == 31 ? kTileW : -(1 << 20));   // halo pixel of this lane, relative to the strip
    // (the 16-byte chunk of channels 8..15 of every slab pixel stays zero: k-step 0 reads 16 channels)
    for (int sl = 0; sl < P.a_slots; ++sl)
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const uint32_t p = lane + 32u * j;
        if (p < static_cast<uint32_t>(kBoxW)) sts128(a_base + sl * kASlotBytes + p * 128u + ((1u ^ (p & 7u)) << 4), 0u, 0u, 0u, 0u);
      }
    pdl_wait();   // the frames (and src_out's last readers) belong to earlier work
    uint32_t as = 0, aph = 0;
    int u = u0, rowc = 0;
    Band b;
    SrcRow row_next;
    bool have_next = false;
    while (next_band(P, u, u1, b)) {
      const int r0 = b.yb > 0 ? b.yb - 1 : b.yb, r1 = b.ye < P.H ? b.ye : b.ye - 1;
      const int n_abs = b.n + P.n_in0;   // (clip plans only: BSVD streams convert their frames in a layout step)
      const int xs = b.strip * kTileW, x4 = xs + 4 * lane;
      have_next = false;
      constexpr int kAhead = 8;   // rows between the L2 prefetch and the load
      if (dw == 0 && lane < 4 * kAhead && r0 + (lane >> 2) <= r1) src_prefetch_row(P, n_abs, r0 + (lane >> 2), xs, lane & 3);
      for (int r = r0; r <= r1; ++r, ++rowc) {
        if (dw == (r & 1) && r + kAhead <= r1) src_prefetch_row(P, n_abs, r + kAhead, xs, lane);
        if (rowc % kStreamSrcWarps != dw) {
          for (int kb = 0; kb < P.nkb; ++kb)
            if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
          continue;
        }
        const bool trow = trace != nullptr && dw == 0 && lane == 0 && rowc < 16;
        long long* const trw = trace + 96 + 2 * (rowc >> 1);
        if (trow) trw[0] = clock64();
        const SrcRow row = have_next ? row_next : src_load_row(P, n_abs, r, x4, xs + src_xe_off);
        have_next = r + kStreamSrcWarps <= r1;
        if (have_next) row_next = src_load_row(P, n_abs, r + kStreamSrcWarps, x4, xs + src_xe_off);
        SrcPix pix[5];
#pragma unroll
        for (int i = 0; i < 4; ++i) pix[i] = src_decode(P, src_px(P, row, i));
        pix[4] = src_decode(P, src_px_extra(row));
        if (r >= b.yb && r < b.ye && x4 < P.W) {   // this CTA's own rows: the decoded pixels for the DenBlock's residual
          const size_t off = ((static_cast<size_t>(n_abs) * P.H + r) * P.W + x4) * 16;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            *reinterpret_cast<uint4*>(P.src_out + off + 16 * i) = make_uint4(pix[i].hi[0], pix[i].hi[1], 0u, 0u);
            if (P.src_out_lo != nullptr) *reinterpret_cast<uint4*>(P.src_out_lo + off + 16 * i) = make_uint4(pix[i].lo[0], pix[i].lo[1], 0u, 0u);
          }
        }
        if (trow) trw[1] = clock64();
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait_u(a_empty + 8 * as, aph ^ 1);
          const uint32_t slab = a_base + as * kASlotBytes;
          const bool low = P.a_tm[kb] != 0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t p = 1u + 4u * lane + i;
            sts128(slab + p * 128u + ((p & 7u) << 4), low ? pix[i].lo[0] : pix[i].hi[0], low ? pix[i].lo[1] : pix[i].hi[1], 0u, 0u);
          }
          if (lane == 0 || lane == 31) {
            const uint32_t p = lane == 0 ? 0u : static_cast<uint32_t>(kBoxW - 1);
            sts128(slab + p * 128u + ((p & 7u) << 4), low ? pix[4].lo[0] : pix[4].hi[0], low ? pix[4].lo[1] : pix[4].hi[1], 0u, 0u);
          }
          fence_proxy_async();   // generic-proxy writes -> visible to the tensor pipe's operand reads
          __syncwarp();
          if (lane == 0) mbar_arrive(a_full + 8 * as);
          if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
        }
      }
    }
  } else {
    // ======================================================= epilogue (warps 2..9)
    const Epilogue& E = P.ep;
    const int ew = warp - 2;
    const int qd = warp & 3;       // TMEM lane quarter this warp may access
    const int par = ew >> 2;       // this warp takes the CTA's output rows with (row counter & 1) == par
    const int m = qd * 32 + lane;  // accumulator row == pixel inside the strip
    const uint32_t stage = stage_base + static_cast<uint32_t>(ew) * stage_stride;
    const bool split_store = P.fast_store == 3;
    const bool bf16 = E.is_bf16 != 0;
    const bool fast = P.fast_store != 0;
    const uint64_t pol_out = l2_policy(P.l2_out);
    // Specialised epilogue arithmetic of the fast path.  The general form decides activation kind, slope source,
    // alpha, residuals and 16-bit type per 8-channel group (about 20 instructions per value); the three shapes the
    // nets actually use are 2-4 instructions per value:
    //   1 LeakyReLU with a constant slope in [0, 1], no residual      (RDB conv1-4, upsampling convs)
    //   2 PReLU with per-channel slopes, no residual                  (SRVGG body)
    //   3 no activation, alpha folded into the weights, 0-2 residuals (RDB conv5, conv_body)
    //   4 ReLU6, no residual                                          (BSVD body)
    int emode = 0;
    if (fast && !bf16 && E.alpha == 1.0f) {
      if (E.act == kActPRelu && E.slope == nullptr && E.res1 == nullptr && E.res2 == nullptr && E.slope_const >= 0.f &&
          E.slope_const <= 1.f)
        emode = 1;
      else if (E.act == kActPRelu && E.slope != nullptr && E.res1 == nullptr && E.res2 == nullptr)
        emode = 2;
      else if (E.act == kActNone)
        emode = 3;
      else if (E.act == kActRelu6 && E.res1 == nullptr && E.res2 == nullptr)
        emode = 4;
    }
    int s = 0, k = 0, q = 0;
    int u = u0;
    Band b;
    const int upc = P.n_img * P.strips * P.H;  // units (output rows of 128 pixels) per chunk
    // Writes the bias row of `chunk_` into accumulator slot s_ (this warp's 32 TMEM lanes) and hands the slot to
    // the MMA stream: every MMA accumulates, the slot's initial value IS the bias (exact fp32).
    auto init_slot = [&](int s_, int chunk_) {
      const uint32_t ta = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + static_cast<uint32_t>(s_ * NOUT);
      const uint32_t ba = bias_base + static_cast<uint32_t>(chunk_ * NOUT) * 4u;
      if (!kBiasMMA) {
#pragma unroll
        for (int c = 0; c < NOUT; c += 16) {
          uint32_t bv[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) lds128(ba + (c + 4 * i) * 4u, bv[4 * i], bv[4 * i + 1], bv[4 * i + 2], bv[4 * i + 3]);
          tmem_st16p(ta + c, bv);
        }
        tmem_st_wait();
      }
      tcgen05_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + 8 * s_);
    };
    // first use of every slot (output rows u0 .. u0+S-1; this warp's parity group)
    for (int q0 = par; q0 < S && u0 + q0 < u1; q0 += 2) init_slot(q0, (u0 + q0) / upc);
    pdl_wait();  // residual loads and output stores touch tensors of the previous kernel
    if (P.discard_ptr != nullptr) {
      // the previous dense block's x1..x4 (and x) are dead once its conv5 has completed: drop their dirty lines from
      // L2 instead of letting them be written back to HBM (4 GB per 720p frame of pure write traffic otherwise)
      const int64_t per = (P.discard_npx + gridDim.x - 1) / gridDim.x;
      const int64_t p0 = per * blockIdx.x, p1 = p0 + per < P.discard_npx ? p0 + per : P.discard_npx;
      uint8_t* const db = reinterpret_cast<uint8_t*>(P.discard_ptr);
      for (int64_t p = p0 + (ew * 32 + lane); p < p1; p += kStreamEpiWarps * 32) {
        uint8_t* const px = db + p * P.discard_pitch_bytes;
#pragma unroll
        for (int l = 0; l < 3; ++l)
          if ((P.discard_mask >> l) & 1u) asm volatile("discard.global.L2 [%0], 128;" ::"l"(px + l * 128) : "memory");
      }
    }
    while (next_band(P, u, u1, b)) {
      const int ax = b.strip * kTileW + m;
      const bool valid = ax < P.W;
      int mask_h = 0x7fffffff;   // crop atlases: rows of this thread's pixel column that lie inside a crop of image b.n
      if (P.mask_hw != nullptr) {
        const int32_t* mt = P.mask_hw + static_cast<size_t>(b.n) * kMaskStride;
        const int cnt = __ldg(mt);
        const int sh = P.mask_shift;
        mask_h = 0;
        for (int k = 0; k < cnt; ++k) {
          const int x0 = __ldg(mt + 1 + 3 * k), w = __ldg(mt + 2 + 3 * k), h = __ldg(mt + 3 + 3 * k);
          const int cx0 = sh >= 0 ? x0 << sh : x0 >> -sh, cw = sh >= 0 ? w << sh : w >> -sh, chh = sh >= 0 ? h << sh : h >> -sh;
          if (ax >= cx0 && ax < cx0 + cw) mask_h = chh;
        }
      }
      for (int y = b.yb; y < b.ye; ++y, ++q) {
        if ((q & 1) == par) {
          // residual prefetch (fast path): issued before the accumulator wait so the latency is hidden
          uint4 r1v[NOUT / 8], r2v[NOUT / 8];
          constexpr bool kPs2 = NOUT <= 32;          // (the planner uses the PixelShuffle(2) fast store with chunks <= 32 only)
          uint4 r1l[kPs2 ? NOUT / 8 : 1];            // split precision + PixelShuffle(2): low halves of the skip tensor
          const int nr1 = ring_n(P, b.n, P.ring_res1);
          const size_t pix1 = (static_cast<size_t>(nr1) * E.out_h + y) * E.out_w + ax;
          const bool has_r1 = fast && E.res1 != nullptr, has_r2 = fast && E.res2 != nullptr;
          // PixelShuffle(2) fast store: this chunk is (part of) sub-pixel phase ab of the shuffled tensor (channels
          // pre-permuted to (a, b, c)); E.out_h / E.out_w are the shuffled sizes
          int ps_ab = 0, ps_c0 = 0;
          const bool ps2 = kPs2 && P.ps2 != 0;
          if (ps2) {
            const int cq = E.cout >> 2;
            ps_ab = (b.chunk * NOUT) / cq;
            ps_c0 = b.chunk * NOUT - ps_ab * cq;
          }
          if (ps2 && has_r1 && valid) {
            const size_t po = (static_cast<size_t>(nr1) * E.out_h + 2 * y + (ps_ab >> 1)) * E.out_w + 2 * ax + (ps_ab & 1);
            const uint16_t* const rb = reinterpret_cast<const uint16_t*>(E.res1) + po * E.res1_pitch + E.res1_coff + ps_c0;
#pragma unroll
            for (int j = 0; j < NOUT / 8; ++j) r1v[j] = reinterpret_cast<const uint4*>(rb)[j];
            if (E.res1_lo_off != 0) {
#pragma unroll
              for (int j = 0; j < NOUT / 8; ++j) r1l[j] = reinterpret_cast<const uint4*>(rb + E.res1_lo_off)[j];
            }
          } else if (has_r1 && valid) {
            if (E.res1_nch > 0) {
              // residual on the first res1_nch (<= 8) channels of the conv only (BSVD none_minus, bsvd/model.py:436-442):
              // one 16-byte load for channel group 0 of chunk 0, the other channels' halves masked to +0
#pragma unroll
              for (int j = 0; j < NOUT / 8; ++j) r1v[j] = make_uint4(0u, 0u, 0u, 0u);
              if (b.chunk == 0) {
                uint4 t = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(E.res1) + pix1 * E.res1_pitch + E.res1_coff);
                const int nch = E.res1_nch;
                t.x &= (nch > 0 ? 0xFFFFu : 0u) | (nch > 1 ? 0xFFFF0000u : 0u);
                t.y &= (nch > 2 ? 0xFFFFu : 0u) | (nch > 3 ? 0xFFFF0000u : 0u);
                t.z &= (nch > 4 ? 0xFFFFu : 0u) | (nch > 5 ? 0xFFFF0000u : 0u);
                t.w &= (nch > 6 ? 0xFFFFu : 0u) | (nch > 7 ? 0xFFFF0000u : 0u);
                r1v[0] = t;
              }
            } else {
              const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(E.res1) + pix1 * E.res1_pitch + E.res1_coff + b.chunk * NOUT);
#pragma unroll
              for (int j = 0; j < NOUT / 8; ++j) r1v[j] = rp[j];
            }
          }
          if (has_r2 && valid) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(E.res2) + ((static_cast<size_t>(ring_n(P, b.n, P.ring_res2)) * E.out_h + y) * E.out_w + ax) * E.res2_pitch + E.res2_coff + b.chunk * NOUT);
#pragma unroll
            for (int j = 0; j < NOUT / 8; ++j) r2v[j] = rp[j];
          }
          const bool trow = trace != nullptr && warp == 2 && lane == 0 && q < 16;
          long long* const trw = trace + 80 + 4 * (q >> 1);
          if (trow) trw[0] = clock64();
          mbar_wait_u(acc_full + 8 * s, k & 1);
          tcgen05_after_sync();
          if (trow) trw[1] = clock64();
          if (warp == 2 && q == 0) SS4K_TRACE(5);
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + static_cast<uint32_t>(s * NOUT);
          uint32_t raw[NOUT];
#pragma unroll
          for (int c = 0; c < NOUT; c += 16) tmem_ld16p(taddr + c, &raw[c]);
          tmem_ld_wait();
          if (y >= mask_h) {   // outside every crop: bias included, every store path starts from raw
#pragma unroll
            for (int c = 0; c < NOUT; ++c) raw[c] = 0u;
          }
          {
            // slot drained: re-initialise it with the bias of the output row that reuses it (S rows ahead in this
            // CTA's unit order, possibly the next chunk) and release it to the MMA stream
            const int ut = u - (b.ye - y) + S;
            if (ut < u1) init_slot(s, ut / upc);
          }
          if (trow) trw[2] = clock64();
          if (!(P.dbg_flags & 4)) {
            if (fast) {
              // ---- activation, residuals, 16-bit pack into the warp's swizzled staging tile, TMA store
              if (lane == 0) bulk_wait_read0();  // this warp's previous store has finished reading the tile
              __syncwarp();
              const uint32_t srow = stage + lane * (NOUT * 2u);
              // swizzled 16-byte chunk position inside the [32 pixels][NOUT] tile (matches tmO's swizzle mode)
              const uint32_t sxor = NOUT == 64 ? (lane & 7u) : (NOUT == 32 ? ((lane >> 1) & 3u) : (NOUT == 16 ? ((lane >> 2) & 1u) : 0u));
              auto h2 = [](float a, float c) -> uint32_t {
                const __half2 h = __floats2half2_rn(a, c);
                return *reinterpret_cast<const uint32_t*>(&h);
              };
              if (emode == 1) {
                const float sl = E.slope_const;
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  float v[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float a = __uint_as_float(raw[8 * j + i]);
                    v[i] = fmaxf(a, a * sl);  // == a >= 0 ? a : a * sl for 0 <= sl <= 1
                  }
                  sts128(srow + ((static_cast<uint32_t>(j) ^ sxor) << 4), h2(v[0], v[1]), h2(v[2], v[3]), h2(v[4], v[5]), h2(v[6], v[7]));
                }
              } else if (emode == 2) {
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  const float4* sp = reinterpret_cast<const float4*>(E.slope + b.chunk * NOUT + 8 * j);
                  const float4 sa = __ldg(sp), sb = __ldg(sp + 1);
                  const float sl[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
                  float v[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float a = __uint_as_float(raw[8 * j + i]);
                    v[i] = fmaf(fminf(a, 0.f), sl[i], fmaxf(a, 0.f));
                  }
                  sts128(srow + ((static_cast<uint32_t>(j) ^ sxor) << 4), h2(v[0], v[1]), h2(v[2], v[3]), h2(v[4], v[5]), h2(v[6], v[7]));
                }
              } else if (split_store) {
                // split precision (BSVD, SS4K_ACT_F16_SPLIT): value = hi + lo with hi = fp16(v), lo = fp16(v - hi); ReLU6 or
                // linear; a residual only as the skip add of a PixelShuffle(2) conv (the planner sends everything else
                // through the specialised / general per-thread paths)
                const bool relu6 = E.act == kActRelu6;
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  uint32_t hi[4], lo[4];
                  const uint32_t rh4[4] = {r1v[j].x, r1v[j].y, r1v[j].z, r1v[j].w};
                  const uint4 rlq = r1l[kPs2 ? j : 0];
                  const uint32_t rl4[4] = {rlq.x, rlq.y, rlq.z, rlq.w};
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    float a = __uint_as_float(raw[8 * j + 2 * i]), c = __uint_as_float(raw[8 * j + 2 * i + 1]);
                    if (relu6) { a = fminf(fmaxf(a, 0.f), 6.f); c = fminf(fmaxf(c, 0.f), 6.f); }
                    if (kPs2 && has_r1) {   // skip add of the PixelShuffle(2) convs: (v + hi) + lo, as the other store paths
                      const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&rh4[i]));
                      a += fh.x; c += fh.y;
                      if (E.res1_lo_off != 0) {
                        const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&rl4[i]));
                        a += fl.x; c += fl.y;
                      }
                    }
                    const __half2 h = __floats2half2_rn(a, c);
                    const float2 back = __half22float2(h);
                    hi[i] = *reinterpret_cast<const uint32_t*>(&h);
                    lo[i] = h2(a - back.x, c - back.y);
                  }
                  const uint32_t off = (static_cast<uint32_t>(j) ^ sxor) << 4;
                  sts128(srow + off, hi[0], hi[1], hi[2], hi[3]);
                  sts128(srow + kStageWarp + off, lo[0], lo[1], lo[2], lo[3]);
                }
              } else if (emode == 4) {
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  float v[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] = fminf(fmaxf(__uint_as_float(raw[8 * j + i]), 0.f), 6.f);
                  sts128(srow + ((static_cast<uint32_t>(j) ^ sxor) << 4), h2(v[0], v[1]), h2(v[2], v[3]), h2(v[4], v[5]), h2(v[6], v[7]));
                }
              } else if (emode == 3) {
                const float b1 = E.beta1, b2 = E.beta2;
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  float v[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(raw[8 * j + i]);
                  if (has_r1) {
                    const uint32_t w4[4] = {r1v[j].x, r1v[j].y, r1v[j].z, r1v[j].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
                      v[2 * i] = fmaf(b1, f.x, v[2 * i]);
                      v[2 * i + 1] = fmaf(b1, f.y, v[2 * i + 1]);
                    }
                  }
                  if (has_r2) {
                    const uint32_t w4[4] = {r2v[j].x, r2v[j].y, r2v[j].z, r2v[j].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
                      v[2 * i] = fmaf(b2, f.x, v[2 * i]);
                      v[2 * i + 1] = fmaf(b2, f.y, v[2 * i + 1]);
                    }
                  }
                  sts128(srow + ((static_cast<uint32_t>(j) ^ sxor) << 4), h2(v[0], v[1]), h2(v[2], v[3]), h2(v[4], v[5]), h2(v[6], v[7]));
                }
              } else
#pragma unroll
              for (int j = 0; j < NOUT / 8; ++j) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(raw[8 * j + i]);
                if (E.act == kActPRelu) {
                  if (E.slope == nullptr) {
                    const float sl = E.slope_const;
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = v[i] >= 0.f ? v[i] : v[i] * sl;
                  } else {
                    const float4* sp = reinterpret_cast<const float4*>(E.slope + b.chunk * NOUT + 8 * j);
                    const float4 sa = __ldg(sp), sb = __ldg(sp + 1);
                    const float sl[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = v[i] >= 0.f ? v[i] : v[i] * sl[i];
                  }
                } else if (E.act == kActRelu6) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] = fminf(fmaxf(v[i], 0.f), 6.f);
                }
                if (E.alpha != 1.0f) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] *= E.alpha;
                }
                if (has_r1) {
                  const uint32_t w4[4] = {r1v[j].x, r1v[j].y, r1v[j].z, r1v[j].w};
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const float2 f = unpack2(w4[i], bf16);
                    v[2 * i] = fmaf(E.beta1, f.x, v[2 * i]);
                    v[2 * i + 1] = fmaf(E.beta1, f.y, v[2 * i + 1]);
                  }
                }
                if (has_r2) {
                  const uint32_t w4[4] = {r2v[j].x, r2v[j].y, r2v[j].z, r2v[j].w};
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const float2 f = unpack2(w4[i], bf16);
                    v[2 * i] = fmaf(E.beta2, f.x, v[2 * i]);
                    v[2 * i + 1] = fmaf(E.beta2, f.y, v[2 * i + 1]);
                  }
                }
                // swizzled 16-byte chunk position inside the [32 pixels][NOUT] tile (matches tmO's swizzle mode)
                uint32_t pj;
                if (NOUT == 64) pj = static_cast<uint32_t>(j) ^ (lane & 7u);
                else if (NOUT == 32) pj = static_cast<uint32_t>(j) ^ ((lane >> 1) & 3u);
                else if (NOUT == 16) pj = static_cast<uint32_t>(j) ^ ((lane >> 2) & 1u);
                else pj = static_cast<uint32_t>(j);
                sts128(stage + lane * (NOUT * 2u) + pj * 16u, pack2(v[0], v[1], bf16), pack2(v[2], v[3], bf16),
                       pack2(v[4], v[5], bf16), pack2(v[6], v[7], bf16));
              }
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) {
                if (P.fast_store == 2) {
#pragma unroll
                  for (int ab = 0; ab < 4; ++ab)
                    tma_store_5d(&P.tmO, stage, b.chunk * NOUT, ab & 1, b.strip * kTileW + qd * 32, ab >> 1, ((b.n + P.n_out0) & P.ring_out) * P.H + y, pol_out);
                } else if (ps2) {
                  tma_store_5d(&P.tmO, stage, ps_c0, ps_ab & 1, b.strip * kTileW + qd * 32, ps_ab >> 1, ((b.n + P.n_out0) & P.ring_out) * P.H + y, pol_out);
                  if (split_store) tma_store_5d(&P.tmO2, stage + kStageWarp, ps_c0, ps_ab & 1, b.strip * kTileW + qd * 32, ps_ab >> 1, ((b.n + P.n_out0) & P.ring_out) * P.H + y, pol_out);
                } else {
                  tma_store_4d(&P.tmO, stage, b.chunk * NOUT, b.strip * kTileW + qd * 32, y, (b.n + P.n_out0) & P.ring_out, pol_out);
                  if (split_store) tma_store_4d(&P.tmO2, stage + kStageWarp, b.chunk * NOUT, b.strip * kTileW + qd * 32, y, (b.n + P.n_out0) & P.ring_out, pol_out);
                }
                bulk_commit();
              }
            } else if (NOUT == 16 && E.out_mode == kOutNV12) {
              if constexpr (NOUT == 16) {
                const ImgAt I = ring_img(P, b.n);
                // NV12 frame store (RRDBNet's conv_last, out_fmt SS4K_FMT_NV12): the bytes of the kOutU8NHWC path, converted
                // with rgb_to_nv12_kernel's integer arithmetic (elementwise.cu).  Each warp stores its own Y row; the
                // parity-0 warp (row 2j) leaves its horizontal chroma pair sums in shared memory, the parity-1 warp (row
                // 2j+1) adds its own and stores UV row j.  Both warps take the quarter's named barrier once per row pair
                // whatever their `valid` lanes.  Two exchange slots suffice: the parity-0 warp refills slot j & 1 only
                // after the barrier of pair j+1, which the parity-1 warp reaches after it has read pair j's sums.
                // (W % 4 == 0 and strips start at multiples of 128: a 4-pixel word is entirely valid or entirely not.)
                int c8[3];
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                  float f = fminf(fmaxf(__uint_as_float(raw[i]), 0.f), 1.f) * 255.f;
                  if (E.round_u8) f = rintf(f);
                  c8[i] = static_cast<uint8_t>(f);
                }
                const uint32_t yv = static_cast<uint32_t>(16 + ((5983 * c8[0] + 20127 * c8[1] + 2032 * c8[2] + 16384) >> 15));
                uint32_t yw = yv | (__shfl_down_sync(0xffffffffu, yv, 1) << 8);
                yw |= __shfl_down_sync(0xffffffffu, yw, 2) << 16;   // lane 4i: Y of pixels 4i .. 4i+3
                // R, G, B of the pixel pair (lanes 2i, 2i+1) as 10-bit fields: a 2x2 sum is at most 1020
                const uint32_t hs1 = static_cast<uint32_t>(c8[0]) | (static_cast<uint32_t>(c8[1]) << 10) | (static_cast<uint32_t>(c8[2]) << 20);
                const uint32_t hs = hs1 + __shfl_xor_sync(0xffffffffu, hs1, 1);
                uint8_t* const frame = reinterpret_cast<uint8_t*>(E.out) + static_cast<size_t>(I.out) * (E.out_h + (E.out_h >> 1)) * E.out_w;
                const bool st_word = valid && (lane & 3) == 0;
                if (st_word) *reinterpret_cast<uint32_t*>(frame + static_cast<size_t>(y) * E.out_w + ax) = yw;
                const uint32_t xchg = rec_base + kMaxSASlots * kRecWords * 4u +
                                      ((((static_cast<uint32_t>(q) >> 1) & 1u) * 4u + static_cast<uint32_t>(qd)) * 16u + (lane >> 1)) * 4u;
                if (par == 0 && (lane & 1) == 0) asm volatile("st.shared.b32 [%0], %1;" ::"r"(xchg), "r"(hs) : "memory");
                asm volatile("bar.sync %0, 64;" ::"r"(kNv12BarBase + qd) : "memory");
                if (par == 1) {
                  uint32_t s4 = hs;
                  if ((lane & 1) == 0) {
                    uint32_t other;
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(other) : "r"(xchg) : "memory");
                    s4 += other;
                  }
                  const int sr = static_cast<int>(s4 & 0x3FFu), sg = static_cast<int>((s4 >> 10) & 0x3FFu), sb = static_cast<int>(s4 >> 20);
                  const int uu = 128 + ((-3298 * sr - 11094 * sg + 14392 * sb + 65536) >> 17);
                  const int vv = 128 + ((14392 * sr - 13073 * sg - 1319 * sb + 65536) >> 17);
                  uint32_t uvw = (static_cast<uint32_t>(uu) & 0xFFu) | ((static_cast<uint32_t>(vv) & 0xFFu) << 8);
                  uvw |= __shfl_down_sync(0xffffffffu, uvw, 2) << 16;   // lane 4i: U, V of pairs 2i, 2i+1
                  if (st_word) *reinterpret_cast<uint32_t*>(frame + static_cast<size_t>(E.out_h + (y >> 1)) * E.out_w + ax) = uvw;
                }
              }
            } else if (NOUT == 16 && E.out_mode == kOutU8NHWC && E.cout == 3 && E.act == kActNone && E.alpha == 1.0f &&
                       E.res1 == nullptr && E.res2 == nullptr && __all_sync(0xffffffffu, valid)) {
              // uint8 RGB frame store (last conv of the nets): the warp's 32 pixels are 96 contiguous bytes; assemble
              // them into 24 words with shuffles instead of three strided byte stores per thread
              uint32_t px = 0;
#pragma unroll
              for (int i = 0; i < 3; ++i) {
                float f = fminf(fmaxf(__uint_as_float(raw[i]), 0.f), 1.f) * 255.f;
                if (E.round_u8) f = rintf(f);
                px |= static_cast<uint32_t>(static_cast<uint8_t>(f)) << (8 * i);
              }
              const int p0 = (4 * lane) / 3, sh = 4 * lane - 3 * p0;  // word `lane` starts `sh` bytes into pixel p0
              const uint32_t lo = __shfl_sync(0xffffffffu, px, p0 & 31), hi = __shfl_sync(0xffffffffu, px, (p0 + 1) & 31);
              const uint64_t two = static_cast<uint64_t>(lo) | (static_cast<uint64_t>(hi) << 24);
              if (lane < 24) {
                const ImgAt I = ring_img(P, b.n);
                const size_t pix0 = (static_cast<size_t>(I.out) * E.out_h + y) * E.out_w + b.strip * kTileW + qd * 32;
                reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(E.out) + pix0 * 3)[lane] = static_cast<uint32_t>(two >> (8 * sh));
              }
            } else if (NOUT == 16 && (E.out_mode == kOutNCHWF16 || E.out_mode == kOutNCHWF32) && E.cout <= 4 &&
                       E.act == kActNone && E.alpha == 1.0f && E.res2 == nullptr && !bf16) {
              // few-channel planar output (last conv of RRDBNet / BSVD at the model boundary, optional residual on the
              // first res1_nch channels: BSVD none_minus, bsvd/model.py:436-442): one coalesced store per channel
              if (valid) {
                const ImgAt I = ring_img(P, b.n);
                const size_t plane = static_cast<size_t>(E.out_h) * E.out_w;
                const size_t o0 = static_cast<size_t>(I.out) * E.cout * plane + static_cast<size_t>(y) * E.out_w + ax;
                const uint16_t* rp = E.res1 != nullptr ? reinterpret_cast<const uint16_t*>(E.res1) + pix1 * E.res1_pitch + E.res1_coff : nullptr;
                const int nres = E.res1 == nullptr ? 0 : (E.res1_nch > 0 ? E.res1_nch : E.cout);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                  if (c < E.cout) {
                    float v = __uint_as_float(raw[c]);
                    if (c < nres) {
                      // (split precision: + the residual's low half; same association as epilogue_chunk)
                      float r = E.beta1 * __half2float(*reinterpret_cast<const __half*>(rp + c));
                      if (E.res1_lo_off != 0) r = fmaf(E.beta1, __half2float(*reinterpret_cast<const __half*>(rp + c + E.res1_lo_off)), r);
                      v += r;
                    }
                    if (E.out_mode == kOutNCHWF16) reinterpret_cast<__half*>(E.out)[o0 + c * plane] = __float2half_rn(v);
                    else reinterpret_cast<float*>(E.out)[o0 + c * plane] = v;
                  }
                }
              }
            } else if (NOUT == 48 && E.out_mode == kOutPSNCHWF16 && E.ps_r == 4 && E.cout == 48 && E.act == kActNone &&
                       E.alpha == 1.0f && E.res1 == nullptr && E.res2 == nullptr && !bf16) {
              // PixelShuffle(4) into half NCHW (+ nearest-upsampled base image): SRVGGNetCompact's last conv
              // (factory.py:69-82).  Conv channel c*16 + a*4 + b of pixel (y, x) is out[n, c, 4y + a, 4x + b]: for one
              // (c, a) a thread owns 4 consecutive output pixels (8 bytes) and a warp 256 contiguous bytes.
              if (valid) {
                const ImgAt I = ring_img(P, b.n);
                const size_t pixi = (static_cast<size_t>(I.out) * E.out_h + y) * E.out_w + ax;
                const int OH = 4 * E.out_h, OW = 4 * E.out_w;
                __half* const o = reinterpret_cast<__half*>(E.out);
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                  float base = 0.f;
                  if (E.base != nullptr)
                    base = __half2float(reinterpret_cast<const __half*>(E.base)[pixi * E.base_pitch + c]);
#pragma unroll
                  for (int a4 = 0; a4 < 4; ++a4) {
                    const int ch = c * 16 + a4 * 4;
                    const __half2 lo = __floats2half2_rn(__uint_as_float(raw[ch]) + base, __uint_as_float(raw[ch + 1]) + base);
                    const __half2 hi = __floats2half2_rn(__uint_as_float(raw[ch + 2]) + base, __uint_as_float(raw[ch + 3]) + base);
                    uint2 w2;
                    w2.x = *reinterpret_cast<const uint32_t*>(&lo);
                    w2.y = *reinterpret_cast<const uint32_t*>(&hi);
                    const size_t oi = ((static_cast<size_t>(I.out) * 3 + c) * OH + (4 * y + a4)) * OW + 4 * static_cast<size_t>(ax);
                    *reinterpret_cast<uint2*>(o + oi) = w2;
                  }
                }
              }
            } else if ((E.out_mode == kOutNHWC || E.out_mode == kOutPS2NHWC) && !E.up2_store && E.alpha == 1.0f &&
                       E.res2 == nullptr && E.res1_nch <= 8 && !bf16 &&
                       (E.act == kActRelu6 || E.act == kActNone) && (E.res1 == nullptr || E.beta1 == 1.0f)) {
              // BSVD stores (bsvd/model.py:43-52, 231-323): ReLU6 or linear, optional PixelShuffle(2) (weights'
              // output channels pre-permuted to (a, b, c)), optional skip add at the output pixel, optional temporal-
              // shift scatter (channels [0, fold) go to frame t-1's tensor, [fold, 2 fold) to frame t+1's).  Same
              // arithmetic as epilogue_chunk, decided once per 8-channel group instead of per value.
              if (valid) {
                const ImgAt I = ring_img(P, b.n);
                const int t = I.t;
                const int cq = E.cout >> 2;
                const bool ps2 = E.out_mode == kOutPS2NHWC;
                const bool relu6 = E.act == kActRelu6;
                uint16_t* const o16 = reinterpret_cast<uint16_t*>(E.out);
#pragma unroll
                for (int j = 0; j < NOUT / 8; ++j) {
                  const int ch0 = b.chunk * NOUT + 8 * j;
                  if (ch0 >= E.cout) break;  // padded output channels
                  int oy = y, ox = ax, oc = ch0;
                  if (ps2) {
                    const int ab = ch0 / cq;
                    oc = ch0 - ab * cq;
                    oy = 2 * y + (ab >> 1);
                    ox = 2 * ax + (ab & 1);
                  }
                  const size_t po = (static_cast<size_t>(I.out) * E.out_h + oy) * E.out_w + ox;
                  const size_t po1 = (static_cast<size_t>(I.res1) * E.out_h + oy) * E.out_w + ox;
                  float v[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float a = __uint_as_float(raw[8 * j + i]);
                    v[i] = relu6 ? fminf(fmaxf(a, 0.f), 6.f) : a;
                  }
                  if (E.res1 != nullptr && (E.res1_nch == 0 || oc == 0)) {
                    // (split precision: the residual tensor has a low-half twin res1_lo_off elements further on;
                    //  res1_nch > 0: only the first channels take part -- BSVD none_minus, model.py:436-442)
                    const uint16_t* const rp = reinterpret_cast<const uint16_t*>(E.res1) + po1 * E.res1_pitch + E.res1_coff + oc;
                    const uint4 r = *reinterpret_cast<const uint4*>(rp);
                    const uint32_t w4[4] = {r.x, r.y, r.z, r.w};
                    float rs[8];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
                      rs[2 * i] = f.x;
                      rs[2 * i + 1] = f.y;
                    }
                    float rl[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                    if (E.res1_lo_off != 0) {
                      const uint4 q = *reinterpret_cast<const uint4*>(rp + E.res1_lo_off);
                      const uint32_t l4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                      for (int i = 0; i < 4; ++i) {
                        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&l4[i]));
                        rl[2 * i] = f.x;
                        rl[2 * i + 1] = f.y;
                      }
                    }
                    if (E.res1_nch > 0) {
#pragma unroll
                      for (int i = 0; i < 8; ++i)
                        if (i < E.res1_nch) v[i] += (E.res1_lo_off != 0 ? rs[i] + rl[i] : rs[i]);
                    } else {
#pragma unroll
                      for (int i = 0; i < 8; ++i) {
                        v[i] += rs[i];
                        if (E.res1_lo_off != 0) v[i] += rl[i];
                      }
                    }
                  }
                  int64_t delta = 0;
                  bool ok = true;
                  if (E.fold > 0) {
                    if (oc < E.fold) { delta = E.off_prev * I.prev; ok = t > 0; }
                    else if (oc < 2 * E.fold) { delta = E.off_next * I.next; ok = t < E.t_count - 1; }
                  }
                  if (ok) {
                    uint4 q4;
                    q4.x = pack2(v[0], v[1], false); q4.y = pack2(v[2], v[3], false); q4.z = pack2(v[4], v[5], false); q4.w = pack2(v[6], v[7], false);
                    const int64_t off = static_cast<int64_t>(po * E.out_pitch + E.out_coff + oc) + delta;
                    *reinterpret_cast<uint4*>(o16 + off) = q4;
                    if (E.out_lo != nullptr) {   // split precision: lo = fp16(v - hi) into the low-half twin
                      const uint32_t h4[4] = {q4.x, q4.y, q4.z, q4.w};
                      uint32_t l4[4];
#pragma unroll
                      for (int i = 0; i < 4; ++i) {
                        const float2 back = __half22float2(*reinterpret_cast<const __half2*>(&h4[i]));
                        l4[i] = pack2(v[2 * i] - back.x, v[2 * i + 1] - back.y, false);
                      }
                      *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(E.out_lo) + off) = make_uint4(l4[0], l4[1], l4[2], l4[3]);
                    }
                  }
                }
              }
            } else if (valid) {
              const ImgAt I = ring_img(P, b.n);
#pragma unroll
              for (int c = 0; c < NOUT; c += 16) {
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(raw[c + i]);
                epilogue_chunk(E, kModeConv3, I, y, ax, 0, b.chunk * NOUT + c, v);
              }
            }
          }
          if (trow) trw[3] = clock64();
        }
        if (++s == S) { s = 0; ++k; }
      }
    }
    if (warp == 2) SS4K_TRACE(6);
    // the staging tiles must have been read before the CTA releases its shared memory; the global writes themselves
    // complete asynchronously and are ordered before the next kernel by grid completion (griddepcontrol.wait there)
    if (fast && lane == 0) { if (P.dbg_flags & 16) bulk_wait0(); else bulk_wait_read0(); }
    if (warp == 2) SS4K_TRACE(7);
  }

  // ---------------------------------------------------------------- teardown
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
    SS4K_TRACE(8);
  }
#undef SS4K_TRACE
}

// ---------------------------------------------------------------- host launcher
cudaError_t conv_stream_prepare() {
  cudaError_t e = cudaFuncSetAttribute(conv3x3_stream_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_stream_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_stream_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_stream_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  return e;
}

template <int NOUT>
static int occupancy_one() {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, conv3x3_stream_kernel<NOUT>, kStreamThreads, kSmemBytes) != cudaSuccess) return 0;
  return n;
}
int conv_stream_max_ctas_per_sm(int nout) {
  switch (nout) {
    case 16: return occupancy_one<16>();
    case 32: return occupancy_one<32>();
    case 48: return occupancy_one<48>();
    case 64: return occupancy_one<64>();
    default: return 0;
  }
}

template <int NOUT>
static cudaError_t launch_one(const StreamParams& p, int grid, cudaStream_t stream, bool pdl) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(p.src_fmt != 0 ? kStreamThreadsMax : kStreamThreads);   // + the frame decoder warps
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, conv3x3_stream_kernel<NOUT>, p);
}

// pdl: programmatic dependent launch -- this kernel may start its prologue (barrier init, TMEM allocation,
// weight loads) while the previous kernel of the stream drains; it waits (griddepcontrol.wait) before it
// touches activations.
cudaError_t conv_stream_launch(const StreamParams& p, int nout, int grid, cudaStream_t stream, bool pdl) {
  switch (nout) {
    case 16: return launch_one<16>(p, grid, stream, pdl);
    case 32: return launch_one<32>(p, grid, stream, pdl);
    case 48: return launch_one<48>(p, grid, stream, pdl);
    case 64: return launch_one<64>(p, grid, stream, pdl);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace ss4k
