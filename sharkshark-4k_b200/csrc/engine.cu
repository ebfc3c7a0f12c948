// Engine: context, weight store, weight packing, plan materialisation (buffers, TMA tensor maps,
// tile configuration, CUDA graph) and the C ABI of include/ss4k.h.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/ss4k.h"
#include "conv_params.h"
#include "elementwise.h"
#include "program.h"

using namespace ss4k;

namespace {

thread_local std::string g_last_error;

std::string fmt(const char* f, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof(buf), f, ap);
  va_end(ap);
  return buf;
}

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

}  // namespace

struct ss4k_ctx {
  int device = 0;
  int nsm = 148;
  int desc_mode = 0;
  std::string err;
  std::map<int, std::map<std::string, HostTensor>> weights;
  EncodeTiledFn encode = nullptr;
  int32_t* err_host = nullptr;  // mapped pinned int[4]: watchdog diagnostics
  int32_t* err_dev = nullptr;
  int64_t launches = 0;
  cudaStream_t stream = nullptr;  // internal stream (ss4k_run_host, graph capture)
};

namespace {

int fail(ss4k_ctx* ctx, int code, const std::string& msg) {
  g_last_error = msg;
  if (ctx) ctx->err = msg;
  return code;
}

#define CK(ctx, call)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(ctx, SS4K_E_CUDA, fmt("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__)); \
  } while (0)

uint16_t f2h(float f, bool bf16) {
  if (bf16) {
    __nv_bfloat16 h = __float2bfloat16_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
  }
  __half h = __float2half_rn(f);
  uint16_t u;
  memcpy(&u, &h, 2);
  return u;
}
float h2f(uint16_t u, bool bf16) {
  if (bf16) {
    __nv_bfloat16 h;
    memcpy(&h, &u, 2);
    return __bfloat162float(h);
  }
  __half h;
  memcpy(&h, &u, 2);
  return __half2float(h);
}

int round_up(int a, int b) { return (a + b - 1) / b * b; }

// ------------------------------------------------------------------------------------------------
// A materialised convolution: packed weights on the device + kernel parameter block + grid.
// Binds the calling thread to the engine's GPU for the duration of an entry point and restores the previous device: the
// caller (a PyTorch process that drives several engines, a worker whose current device is still 0) need not have it set.
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (dev < 0) return;
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != dev && cudaSetDevice(dev) == cudaSuccess) prev = cur;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

struct ConvExec {
  ConvParams p;
  StreamParams sp;      // row-streaming kernel (conv_stream.cu) when `stream` is set
  bool stream = false;
  int nout = 0;         // accumulator slot width of the streaming kernel
  int grid = 0;
  void* d_w = nullptr;
  size_t w_bytes = 0;
  float* d_bias = nullptr;
  float* d_slope = nullptr;
  bool ext_out = false;  // ep.out is the caller's output pointer (patched per run)
  bool src_ext = false;  // sp.src is the caller's input pointer (frame-format source decoded by the producer warp, patched per run)
  size_t src_off = 0;    //   byte offset of the step's first frame in it
  std::string name;
};

struct PackedWeights {
  std::vector<uint16_t> w;  // [(nkb*ntaps)][npad_total][64]
  std::vector<float> bias, slope;
  std::vector<KBlock> kb;
  std::vector<Tap> taps;
  std::vector<uint8_t> mask;  // [nkb][kMaxTaps]
  int nkb = 0, ntaps = 0, nsub = 1, max_dr = 2, npad_total = 0;
};

// effective weight of tap t for (out channel n, in channel c); see DESIGN.md section 4.3
struct TapGeom {
  int ntaps, nsub, max_dr;
};

// Lower OIHW fp32 weights to the kernel's packed K-block/tap layout.
//   W: [cout][cin][3][3]; in_coff/in_pitch describe where the cin channels sit in the source tensor.
std::string pack_weights(const ConvSpec& cs, const HostTensor& W, const HostTensor* B, const HostTensor* S,
                         bool bf16, PackedWeights* out) {
  if (W.shape.size() != 4 || W.shape[0] != cs.cout || W.shape[1] != cs.cin || W.shape[2] != 3 || W.shape[3] != 3)
    return fmt("weight %s has shape [%lld,%lld,..], expected [%d,%d,3,3]", cs.wname.c_str(),
               (long long)(W.shape.size() > 0 ? W.shape[0] : -1), (long long)(W.shape.size() > 1 ? W.shape[1] : -1),
               cs.cout, cs.cin);
  if (B && (int)B->data.size() != cs.cout) return fmt("bias %s has wrong size", cs.bname.c_str());
  if (S && (int)S->data.size() != cs.cout) return fmt("slope %s has wrong size", cs.sname.c_str());
  const int npad = round_up(cs.cout, 16);
  out->npad_total = npad;
  auto w_at = [&](int n, int c, int ky, int kx) -> float {
    const float v = W.data[((static_cast<size_t>(n) * cs.cin + c) * 3 + ky) * 3 + kx];
    return n < cs.neg_first ? -v : v;
  };
  // output-channel permutation (PixelShuffle(2) fused store): packed row (a*2+b)*Cq + c  <-  c*4 + a*2 + b
  std::vector<int> orow(npad, -1);
  for (int n = 0; n < cs.cout; ++n) {
    if (cs.wperm == 1) {
      const int cq = cs.cout / 4;
      const int c = n / 4, ab = n % 4;
      orow[ab * cq + c] = n;
    } else {
      orow[n] = n;
    }
  }
  // taps
  out->taps.clear();
  if (cs.mode == kModeConv3) {
    out->nsub = 1; out->max_dr = 2;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) out->taps.push_back(Tap{(int8_t)ky, (int8_t)kx, 0, 0});
  } else if (cs.mode == kModeUp2) {
    out->nsub = 4; out->max_dr = 2;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        for (int tr = 0; tr < 2; ++tr)
          for (int tc = 0; tc < 2; ++tc)
            out->taps.push_back(Tap{(int8_t)(a + tr), (int8_t)(b + tc), (int8_t)(a * 2 + b), 0});
  } else if (cs.mode == kModeS2) {
    out->nsub = 1; out->max_dr = 1;
    for (int dy = 0; dy < 2; ++dy)
      for (int dx = 0; dx < 2; ++dx) out->taps.push_back(Tap{(int8_t)dy, (int8_t)dx, 0, 0});
  } else {
    return "unknown conv mode";
  }
  out->ntaps = (int)out->taps.size();
  // K blocks: (tmap, c0, p) + which weight half (hi/lo) they multiply with
  struct KB { KBlock kb; int whalf; int cbase; int pa; };  // cbase: channel of W that kb channel 0 maps to
  std::vector<KB> kbs;
  const int nsplit = cs.split ? 3 : 1;
  if (cs.mode == kModeS2) {
    if (cs.in_coff != 0 || cs.in_pitch % 16) return "stride-2 conv needs in_coff == 0 and pitch % 16 == 0";
    const int merged = 2 * cs.in_pitch;
    for (int pa = 0; pa < 2; ++pa)
      for (int c0 = 0; c0 < merged; c0 += 64)
        for (int sp = 0; sp < nsplit; ++sp)
          kbs.push_back(KB{KBlock{sp == 2 ? 1 : 0, c0, pa, 0}, sp == 1 ? 1 : 0, c0, pa});
  } else {
    for (int c0 = 0; c0 < cs.cin; c0 += 64)
      for (int sp = 0; sp < nsplit; ++sp)
        kbs.push_back(KB{KBlock{sp == 2 ? 1 : 0, cs.in_coff + c0, 0, 0}, sp == 1 ? 1 : 0, c0, 0});
  }
  out->nkb = (int)kbs.size();
  if (out->nkb > kMaxKBlocks) return fmt("conv %s needs %d K blocks (max %d)", cs.name.c_str(), out->nkb, kMaxKBlocks);
  out->kb.clear();
  for (auto& k : kbs) out->kb.push_back(k.kb);
  out->mask.assign(static_cast<size_t>(out->nkb) * kMaxTaps, 0);
  out->w.assign(static_cast<size_t>(out->nkb) * out->ntaps * npad * 64, 0);

  static const int up_sets[2][2][3] = {{{0, -1, -1}, {1, 2, -1}}, {{0, 1, -1}, {2, -1, -1}}};
  for (int kbi = 0; kbi < out->nkb; ++kbi) {
    const KB& K = kbs[kbi];
    for (int t = 0; t < out->ntaps; ++t) {
      uint8_t m = 0;
      for (int cc = 0; cc < 64; ++cc) {
        // which weight taps / channel does (kb channel cc, tap t) correspond to
        int wc = -1;
        int kys[3] = {-1, -1, -1}, kxs[3] = {-1, -1, -1};
        if (cs.mode == kModeConv3) {
          wc = K.cbase + cc;
          kys[0] = out->taps[t].dr; kxs[0] = out->taps[t].shift;
        } else if (cs.mode == kModeUp2) {
          wc = K.cbase + cc;
          const int a = out->taps[t].sub >> 1, b = out->taps[t].sub & 1;
          const int tr = out->taps[t].dr - a, tc = out->taps[t].shift - b;
          for (int i = 0; i < 3; ++i) { kys[i] = up_sets[a][tr][i]; kxs[i] = up_sets[b][tc][i]; }
        } else {  // kModeS2: merged channel = pb*pitch + c
          const int mch = K.cbase + cc;
          const int pb = mch / cs.in_pitch;
          const int c = mch - pb * cs.in_pitch;
          const int dy = out->taps[t].dr - 1, dx = out->taps[t].shift - 1;
          const int ky = 2 * dy + K.pa + 1, kx = 2 * dx + pb + 1;
          if (pb < 2 && ky >= 0 && kx >= 0) { wc = c; kys[0] = ky; kxs[0] = kx; }
        }
        if (wc < 0 || wc >= cs.cin) continue;
        bool any = false;
        for (int row = 0; row < npad; ++row) {
          const int n = orow[row];
          if (n < 0) continue;
          float sum = 0.f;
          for (int i = 0; i < 3 && kys[i] >= 0; ++i)
            for (int j = 0; j < 3 && kxs[j] >= 0; ++j) sum += w_at(n, wc, kys[i], kxs[j]);
          const uint16_t hi = f2h(sum, bf16);
          uint16_t val = hi;
          if (K.whalf == 1) val = f2h(sum - h2f(hi, bf16), bf16);
          out->w[((static_cast<size_t>(kbi) * out->ntaps + t) * npad + row) * 64 + cc] = val;
          any = true;
        }
        if (any) m |= static_cast<uint8_t>(1u << (cc / 16));
      }
      out->mask[static_cast<size_t>(kbi) * kMaxTaps + t] = m;
    }
  }
  out->bias.assign(npad, 0.f);
  out->slope.assign(npad, 1.f);
  for (int row = 0; row < npad; ++row) {
    const int n = orow[row];
    if (n < 0) continue;
    if (B) out->bias[row] = n < cs.neg_first ? -B->data[n] : B->data[n];
    out->slope[row] = S ? S->data[n] : cs.const_slope;
  }
  return "";
}


// ------------------------------------------------------------------------------------------------
// Row-streaming kernel (conv_stream.cu): weight layout [chunk][K block][kx][2-ky][NOUT][64 channels],
// i.e. one swizzle-128B tile of 3*NOUT rows per (K block, horizontal tap): the three vertical taps
// are stacked along the MMA N dimension.
struct StreamPacked {
  std::vector<uint16_t> w;
  std::vector<float> bias, slope;
  std::vector<float> bias_f;  // bias with alpha (and the none_minus sign) folded in: initial value of the accumulators
  int nout = 0, chunks = 0, nkb = 0, npad_total = 0, a_slots = 0, acc_slots = 0;
  int bias_row0 = 0;     // rows of weight tiles == first row of the bias tiles (bias-MMA variant)
  float alpha_out = 1.f; // epilogue scale left after folding alpha into weights and bias
  uint8_t nks[kMaxSKB];
  uint8_t src_kb[kMaxSKB];  // 64-channel block of the source tensor read by K block i
  uint8_t src_tm[kMaxSKB];  // 0: the tensor itself (high halves in split mode), 1: its low-half twin
  uint8_t whalf[kMaxSKB];   // 0: weights (high halves), 1: low halves of the weights
  uint8_t wt[kMaxSKB];      // weight tile group read by K block i (split mode: A_hi*W_hi and A_lo*W_hi share W_hi's tiles)
  int nwt = 0;              // distinct weight tile groups per output chunk
  int stride2 = 0, nkx = 3;
  uint8_t ksm[kMaxSKB][2];  // stride 2: k-step masks per (K block, horizontal shift)
  int split_fast = 0;       // split precision with the hi / lo twin staging tiles and two TMA stores (StreamParams::fast_store 3)
};

// Output side of a conv that can leave through the swizzled staging tile + TMA store.
static bool stream_fast_store_ok(const ConvSpec& cs, int nout) {
  if (getenv("SS4K_NO_FAST_STORE") != nullptr || !(nout == 16 || nout == 32 || nout == 64)) return false;
  if (cs.out_buf < 0 || cs.out_coff % 8 || cs.out_pitch % 8 || cs.tshift) return false;
  if (cs.out_mode == kOutPS2NHWC) {
    // PixelShuffle(2) (+ skip add): a chunk must lie inside one sub-pixel phase of the (a, b, c)-permuted channels
    const int cq = cs.cout / 4;
    return getenv("SS4K_NO_PS2_FAST") == nullptr && nout <= 32 && cs.wperm == 1 && cs.cout % 4 == 0 && cq % nout == 0 && cs.act == kActNone &&
           cs.alpha == 1.f && cs.res2_buf < 0 && cs.res1_nch == 0 && (cs.res1_buf < 0 || (cs.beta1 == 1.f && cs.res1_pitch % 8 == 0 && cs.res1_coff % 8 == 0)) &&
           !cs.up2_store && cs.mode == kModeConv3;
  }
  return cs.out_mode == kOutNHWC &&
         (cs.res1_nch == 0 || (cs.res1_nch <= 8 && cs.res1_pitch >= 8 && cs.res1_coff % 8 == 0 && cs.res1_lo_buf < 0));
}
// ... and, for the hi / lo output pair of split precision: ReLU6 or linear, nothing folded behind the activation, no residual
// except the skip add of a PixelShuffle(2) conv
static bool stream_split_fast_ok(const ConvSpec& cs, int nout) {
  const bool ps2 = cs.out_mode == kOutPS2NHWC;
  return cs.out_lo_buf >= 0 && stream_fast_store_ok(cs, nout) && (ps2 || cs.res1_buf < 0) && cs.res2_buf < 0 && !cs.up2_store &&
         (cs.act == kActNone || cs.act == kActRelu6) && cs.alpha == 1.f && getenv("SS4K_NO_SPLIT_FAST") == nullptr;
}

bool stream_config(const ConvSpec& cs, StreamPacked* sp) {
  const bool s2 = cs.mode == kModeS2;
  if (cs.mode != kModeConv3 && !s2) return false;
  if (cs.in_coff % 8 || cs.in_pitch % 8) return false;
  // stride 2 reads the pixel-pair view (2 * pitch channels per pair, 64-channel K blocks): pitch 32 or a multiple of 64
  if (s2 && (cs.in_coff != 0 || (2 * cs.in_pitch) % 64 || cs.cin > cs.in_pitch || cs.in_h % 2 || cs.in_w % 2)) return false;
  if (s2 && getenv("SS4K_NO_STREAM_S2")) return false;
  if (getenv("SS4K_NO_STREAM")) return false;
  if (cs.split && getenv("SS4K_NO_STREAM_SPLIT")) return false;
  const int npad = round_up(cs.cout, 16);
  if (npad * 4 > kStreamBiasBytes) return false;
  // fp16 hi/lo split operands: three K blocks per 64 source channels: A_hi*W_hi, A_hi*W_lo, A_lo*W_hi
  const int nsplit = cs.split ? 3 : 1;
  const int nkb0 = s2 ? 2 * cs.in_pitch / 64 : (cs.cin + 63) / 64;
  const int nkb = nkb0 * nsplit;
  const int nwt = nkb0 * (cs.split ? 2 : 1);   // W_hi (shared by A_hi and A_lo) and W_lo tile groups per source block
  const int nkx = s2 ? 2 : 3;
  if (nkb > kMaxSKB) return false;
  int cand[4], nc = 0;
  if (npad <= 64) cand[nc++] = npad;
  else if (npad % 64 == 0) cand[nc++] = 64;
  if (npad % 32 == 0 && npad > 32) cand[nc++] = 32;
  if (npad > 16) cand[nc++] = 16;
  // a PixelShuffle(2) conv prefers the widest chunk that can still leave through TMA stores (its per-thread store path is
  // the slower one); everything else takes the widest chunk that fits
  bool want_fast = false;
  if (cs.out_mode == kOutPS2NHWC)
    for (int i = 0; i < nc; ++i) want_fast = want_fast || (npad % cand[i] == 0 && stream_fast_store_ok(cs, cand[i]));
  for (int i = 0; i < nc; ++i) {
    const int nout = cand[i];
    if (npad % nout) continue;
    if (want_fast && !stream_fast_store_ok(cs, nout)) continue;
    const int wbytes = nwt * nkx * 3 * nout * 128 + (stream_bias_mma(nout) ? nout * 128 + kStreamOnesBytes : kStreamBiasBytes);
    // epilogue staging tiles (one per epilogue warp; twin tiles for the hi / lo pair of split precision) exist only for
    // convs that leave through TMA stores: the others keep the shared memory for slabs / a wider chunk
    int stage = kStreamEpiWarps * round_up(32 * nout * 2, 1024);
    int left = kSmemBytes - 3072 - wbytes;  // 1 KB alignment slack + barriers, row records, row_ready ring
    int split_fast = 0;
    const bool plain_fast = stream_fast_store_ok(cs, nout) && cs.out_lo_buf < 0;
    if (stream_split_fast_ok(cs, nout) && (left - 2 * stage) / kASlotBytes >= 3) {  // twin tiles only where three slabs still fit
      left -= 2 * stage; split_fast = 1;
    } else if (plain_fast || getenv("SS4K_KEEP_STAGE") != nullptr) {
      left -= stage;
    }
    const int slots = std::min(kMaxSASlots, left / kASlotBytes);
    // a wider chunk is worth it only with enough slabs in flight (experiments: SS4K_MIN_SLOTS)
    static const int min_slots = getenv("SS4K_MIN_SLOTS") ? std::max(3, atoi(getenv("SS4K_MIN_SLOTS"))) : 3;
    if (slots < (nout > 16 ? min_slots : 3)) continue;
    sp->nout = nout; sp->chunks = npad / nout; sp->nkb = nkb; sp->npad_total = npad;
    sp->stride2 = s2 ? 1 : 0; sp->nkx = nkx; sp->nwt = nwt; sp->split_fast = split_fast;
    sp->a_slots = slots; sp->acc_slots = std::min(kMaxAccSlots, kTmemCols / nout) & ~1;  // even: rows alternate between two epilogue warp groups
    for (int kb = 0; kb < nkb; ++kb) {
      const int b0 = kb / nsplit, part = kb % nsplit;
      sp->nks[kb] = static_cast<uint8_t>(s2 ? 4 : (std::min(64, cs.cin - 64 * b0) + 15) / 16);
      sp->src_kb[kb] = static_cast<uint8_t>(b0);
      sp->src_tm[kb] = part == 2 ? 1 : 0;
      sp->whalf[kb] = part == 1 ? 1 : 0;
      sp->wt[kb] = static_cast<uint8_t>(cs.split ? 2 * b0 + (part == 1 ? 1 : 0) : b0);
      sp->ksm[kb][0] = sp->ksm[kb][1] = 0;
      if (s2) {
        // merged channel m = b0*64 + cc of the pair view: half = m / pitch (0 even pixel, 1 odd pixel), c = m % pitch.
        // shift 0 (pair x-1): odd half with kx = 0; shift 1 (pair x): even half kx = 1, odd half kx = 2.
        for (int ks = 0; ks < 4; ++ks) {
          const int m = b0 * 64 + ks * 16;
          const int half = m / cs.in_pitch, c = m % cs.in_pitch;
          if (c >= cs.cin) continue;
          if (half == 1) sp->ksm[kb][0] |= static_cast<uint8_t>(1u << ks);
          sp->ksm[kb][1] |= static_cast<uint8_t>(1u << ks);
        }
      }
    }
    return true;
  }
  return false;
}

// kOutNV12 is stored by the <16> streaming kernel's epilogue (conv_stream.cu); a conv that runs elsewhere writes uint8 RGB
// and the plan converts it (ss4k_plan_create)
bool stream_nv12_ok(const ConvSpec& cs) {
  StreamPacked sp;
  return stream_config(cs, &sp) && sp.nout == 16 && sp.chunks == 1 && cs.cout == 3 && cs.act == kActNone && cs.alpha == 1.f &&
         cs.res1_buf < 0 && cs.res2_buf < 0 && cs.out_h % 2 == 0 && cs.out_w % 4 == 0;
}

std::string pack_weights_stream(const ConvSpec& cs, const HostTensor& W, const HostTensor* B, const HostTensor* S,
                                bool bf16, StreamPacked* out) {
  if (W.shape.size() != 4 || W.shape[0] != cs.cout || W.shape[1] != cs.cin || W.shape[2] != 3 || W.shape[3] != 3)
    return fmt("weight %s has the wrong shape, expected [%d,%d,3,3]", cs.wname.c_str(), cs.cout, cs.cin);
  if (B && (int)B->data.size() != cs.cout) return fmt("bias %s has wrong size", cs.bname.c_str());
  if (S && (int)S->data.size() != cs.cout) return fmt("slope %s has wrong size", cs.sname.c_str());
  const int npad = out->npad_total, nout = out->nout, nkb = out->nkb;
  std::vector<int> orow(npad, -1);
  for (int n = 0; n < cs.cout; ++n) {
    if (cs.wperm == 1) {
      const int cq = cs.cout / 4;
      orow[(n % 4) * cq + n / 4] = n;
    } else {
      orow[n] = n;
    }
  }
  // alpha * act(conv + bias) == act(alpha*conv + alpha*bias) for the positively homogeneous activations
  // (none, PReLU / LeakyReLU): fold alpha into weights and bias so the epilogue does not multiply
  const float fold = (cs.act != kActRelu6) ? cs.alpha : 1.f;
  out->alpha_out = (cs.act != kActRelu6) ? 1.f : cs.alpha;
  // weight tiles, then (bias-MMA variant) one bias tile per chunk: row = output channel, K column 0 = high half,
  // column 1 = low half of the bias (the "ones" operand has 1 there)
  const int nkx = out->nkx;
  const int nwt = out->nwt;
  const size_t wrows = static_cast<size_t>(out->chunks) * nwt * nkx * 3 * nout;
  out->bias_row0 = static_cast<int>(wrows);
  out->w.assign((wrows + (stream_bias_mma(nout) ? npad : 0)) * 64, 0);
  // vertical tap of N block `blk`: stride 1 stacks [ky2 | ky1 | ky0] (block = 2 - ky); stride 2 stacks [ky2 | ky0 | ky1]
  static const int ky_s1[3] = {2, 1, 0}, ky_s2[3] = {2, 0, 1};
  for (int ch = 0; ch < out->chunks; ++ch)
    for (int kb = 0; kb < nkb; ++kb)
      for (int kx = 0; kx < nkx; ++kx)
        for (int blk = 0; blk < 3; ++blk)
          for (int co = 0; co < nout; ++co) {
            const int n = orow[ch * nout + co];
            if (n < 0) continue;
            if (kb > 0 && out->wt[kb] <= out->wt[kb - 1] && out->whalf[kb] == 0 && cs.split) continue;   // A_lo * W_hi: W_hi's tiles are already there
            const size_t row = ((((static_cast<size_t>(ch) * nwt + out->wt[kb]) * nkx + kx) * 3 + blk) * nout + co);
            for (int cc = 0; cc < 64; ++cc) {
              int c, wkx;
              if (out->stride2) {
                const int m = out->src_kb[kb] * 64 + cc;
                const int half = m / cs.in_pitch;
                c = m % cs.in_pitch;
                if (half > 1 || c >= cs.cin) continue;
                if (kx == 0) { if (half == 0) continue; wkx = 0; }   // pair x-1: its odd pixel is input column 2x-1
                else wkx = half == 0 ? 1 : 2;                        // pair x: columns 2x and 2x+1
              } else {
                c = out->src_kb[kb] * 64 + cc;
                if (c >= cs.cin) break;
                wkx = kx;
              }
              const int ky = out->stride2 ? ky_s2[blk] : ky_s1[blk];
              const float wv = (n < cs.neg_first ? -fold : fold) * W.data[((static_cast<size_t>(n) * cs.cin + c) * 3 + ky) * 3 + wkx];
              const uint16_t hi = f2h(wv, bf16);
              out->w[row * 64 + cc] = out->whalf[kb] ? f2h(wv - h2f(hi, bf16), bf16) : hi;
            }
          }
  // the accumulators start from the bias (fp32, written by the epilogue warps with tcgen05.st)
  out->bias_f.assign(npad, 0.f);
  for (int row = 0; row < npad; ++row) {
    const int n = orow[row];
    if (n < 0 || !B) continue;
    out->bias_f[row] = (n < cs.neg_first ? -fold : fold) * B->data[n];
    if (stream_bias_mma(nout)) {
      const uint16_t hi = f2h(out->bias_f[row], bf16);
      out->w[(wrows + row) * 64 + 0] = hi;
      out->w[(wrows + row) * 64 + 1] = f2h(out->bias_f[row] - h2f(hi, bf16), bf16);
    }
  }
  out->bias.assign(npad, 0.f);
  out->slope.assign(npad, 1.f);
  for (int row = 0; row < npad; ++row) {
    const int n = orow[row];
    if (n < 0) continue;
    if (B) out->bias[row] = n < cs.neg_first ? -B->data[n] : B->data[n];
    out->slope[row] = S ? S->data[n] : cs.const_slope;
  }
  return "";
}

// ------------------------------------------------------------------------------------------------
struct TileCfg {
  int R, n_cta, n_chunks, acc_stride, tiles_x, tiles_y, n_tiles;
  int a_slots, a_slot_bytes, a_sub_bytes, w_slots, w_slot_bytes, w_tile_bytes, w_resident;
};

std::string configure_tiles(int desc_mode, int nsm, int n_img, int H, int W, int npad_total, int ntaps,
                            int nsub, int max_dr, int nkb, TileCfg* t) {
  t->n_chunks = (npad_total + 63) / 64;
  if (npad_total % t->n_chunks) return "output channels not divisible into equal chunks";
  t->n_cta = npad_total / t->n_chunks;
  if (t->n_cta % 16) return "chunk width must be a multiple of 16";
  t->acc_stride = round_up(t->n_cta, 32);
  const int max_acc = kAccStageCols / t->acc_stride;
  int rmax = std::min(8, max_acc / nsub);
  if (rmax < 1) return "accumulators do not fit one TMEM stage";
  t->tiles_x = (W + kTileW - 1) / kTileW;
  double best = 1e30;
  int bestR = 1;
  for (int R = 1; R <= rmax; ++R) {
    const int ty = (H + R - 1) / R;
    const long tiles = static_cast<long>(n_img) * ty * t->tiles_x * t->n_chunks;
    const long waves = (tiles + nsm - 1) / nsm;
    const double cost = static_cast<double>(waves) * (R + 0.3 * max_dr + 0.2);
    if (cost < best - 1e-9) { best = cost; bestR = R; }
  }
  t->R = bestR;
  t->tiles_y = (H + t->R - 1) / t->R;
  t->n_tiles = n_img * t->tiles_y * t->tiles_x * t->n_chunks;
  t->w_tile_bytes = t->n_cta * kRowBytes;
  t->w_slot_bytes = ntaps * t->w_tile_bytes;
  t->w_resident = (nkb == 1 && t->n_chunks == 1) ? 1 : 0;
  t->a_sub_bytes = kTileW * kRowBytes;
  t->a_slot_bytes = desc_mode == 2 ? 3 * t->a_sub_bytes : round_up(kBoxW * kRowBytes, 1024);
  const int avail = kSmemBytes - 1024 - 512;
  t->w_slots = t->w_resident ? 1 : 2;
  if (t->w_slots * t->w_slot_bytes + 2 * t->a_slot_bytes > avail) t->w_slots = 1;
  const int left = avail - t->w_slots * t->w_slot_bytes;
  t->a_slots = std::min(kMaxASlots, left / t->a_slot_bytes);
  if (t->a_slots < 2) return "shared memory budget exceeded";
  return "";
}

std::string encode_act_map(ss4k_ctx* ctx, CUtensorMap* tm, void* ptr, int n, int h, int w, int pitch, int mode,
                           bool bf16, int box_w) {
  cuuint64_t dims[5];
  cuuint64_t strides[4];
  const cuuint64_t eb = 2;
  if (mode == kModeS2) {
    if (h % 2 || w % 2) return "stride-2 conv needs even H and W";
    dims[0] = 2 * pitch; dims[1] = w / 2; dims[2] = 2; dims[3] = h / 2; dims[4] = n;
    strides[0] = 2 * pitch * eb;
    strides[1] = static_cast<cuuint64_t>(w) * pitch * eb;
    strides[2] = 2 * static_cast<cuuint64_t>(w) * pitch * eb;
    strides[3] = static_cast<cuuint64_t>(h) * w * pitch * eb;
  } else {
    dims[0] = pitch; dims[1] = w; dims[2] = 1; dims[3] = h; dims[4] = n;
    strides[0] = pitch * eb;
    strides[1] = static_cast<cuuint64_t>(w) * pitch * eb;
    strides[2] = static_cast<cuuint64_t>(w) * pitch * eb;
    strides[3] = static_cast<cuuint64_t>(h) * w * pitch * eb;
  }
  cuuint32_t box[5] = {64, static_cast<cuuint32_t>(box_w), 1, 1, 1};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = ctx->encode(tm, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, ptr,
                           dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fmt("cuTensorMapEncodeTiled(activation) failed: %d", (int)r);
  return "";
}

std::string encode_w_map(ss4k_ctx* ctx, CUtensorMap* tm, void* ptr, int npad_total, int ntiles, int n_cta,
                         int ntaps, bool bf16) {
  cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(npad_total), static_cast<cuuint64_t>(ntiles)};
  cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(npad_total) * 128};
  cuuint32_t box[3] = {64, static_cast<cuuint32_t>(n_cta), static_cast<cuuint32_t>(ntaps)};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = ctx->encode(tm, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, ptr,
                           dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fmt("cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
  return "";
}

void free_conv(ConvExec& c) {
  if (c.d_w) cudaFree(c.d_w);
  if (c.d_bias) cudaFree(c.d_bias);
  if (c.d_slope) cudaFree(c.d_slope);
  c.d_w = nullptr; c.d_bias = nullptr; c.d_slope = nullptr;
}


template <class BufPtr>
void fill_epilogue(const ConvSpec& cs, bool bf16, BufPtr bufptr, float* d_bias, float* d_slope, Epilogue* Ep, bool* ext_out) {
  Epilogue& E = *Ep;
  E.bias = d_bias;
  E.slope = d_slope;
  E.act = cs.act; E.out_mode = cs.out_mode;
  E.alpha = cs.alpha; E.beta1 = cs.beta1; E.beta2 = cs.beta2;
  E.is_bf16 = bf16 ? 1 : 0;
  E.res1 = cs.res1_buf >= 0 ? bufptr(cs.res1_buf) : nullptr;
  E.res2 = cs.res2_buf >= 0 ? bufptr(cs.res2_buf) : nullptr;
  E.res1_pitch = cs.res1_pitch; E.res1_coff = cs.res1_coff;
  E.res2_pitch = cs.res2_pitch; E.res2_coff = cs.res2_coff;
  *ext_out = cs.out_buf == kBufExternalOut;
  E.out = cs.out_buf >= 0 ? bufptr(cs.out_buf) : nullptr;
  E.out_lo = cs.out_lo_buf >= 0 ? bufptr(cs.out_lo_buf) : nullptr;
  E.out2 = cs.out2_buf >= 0 ? bufptr(cs.out2_buf) : nullptr;
  E.out3 = cs.out3_buf >= 0 ? bufptr(cs.out3_buf) : nullptr;
  E.out_pitch = cs.out_pitch; E.out_coff = cs.out_coff;
  E.out_h = cs.out_h; E.out_w = cs.out_w;
  E.cout = cs.cout; E.ps_r = cs.ps_r; E.fold = cs.fold; E.round_u8 = cs.round_u8;
  E.base = cs.base_buf >= 0 ? bufptr(cs.base_buf) : nullptr;
  E.base_pitch = cs.base_pitch;
  E.slope_const = cs.const_slope;
  E.res1_nch = cs.res1_nch;
  E.up2_store = cs.up2_store;
  E.t0 = cs.n0; E.t_count = cs.n_total > 0 ? cs.n_total : cs.n;
  if (cs.n0 > 0) {
    // the kernels index images from 0: a step that starts at frame n0 of the clip gets its tensors' frame n0 as base
    auto adv = [&](const void* p, int64_t frame_elems) { return p ? static_cast<const void*>(reinterpret_cast<const uint16_t*>(p) + cs.n0 * frame_elems) : p; };
    const int64_t fo = static_cast<int64_t>(cs.out_h) * cs.out_w * cs.out_pitch;
    if (cs.out_buf >= 0) { E.out = const_cast<void*>(adv(E.out, fo)); E.out_lo = const_cast<void*>(adv(E.out_lo, fo)); }
    E.res1 = adv(E.res1, static_cast<int64_t>(cs.out_h) * cs.out_w * cs.res1_pitch);
    E.res2 = adv(E.res2, static_cast<int64_t>(cs.out_h) * cs.out_w * cs.res2_pitch);
  }
  E.off_prev = E.off_next = 0;
  E.res1_lo_off = E.res2_lo_off = 0;
  if (cs.res1_buf >= 0 && cs.res1_lo_buf >= 0)
    E.res1_lo_off = reinterpret_cast<const uint16_t*>(bufptr(cs.res1_lo_buf)) - reinterpret_cast<const uint16_t*>(bufptr(cs.res1_buf));
  if (cs.res2_buf >= 0 && cs.res2_lo_buf >= 0)
    E.res2_lo_off = reinterpret_cast<const uint16_t*>(bufptr(cs.res2_lo_buf)) - reinterpret_cast<const uint16_t*>(bufptr(cs.res2_buf));
  if (cs.tshift) {  // clip mode: time == batch index, neighbouring frames are one image stride away
    const int64_t frame = static_cast<int64_t>(cs.out_h) * cs.out_w * cs.out_pitch;
    E.off_prev = -frame; E.off_next = frame;
  } else {
    E.fold = 0;
  }
}

// Row-streaming path: parameter block of conv_stream.cu
template <class BufPtr>
int materialize_stream(ss4k_ctx* ctx, const ConvSpec& cs, const HostTensor& W, const HostTensor* B,
                       const HostTensor* S, bool bf16, StreamPacked& pk, BufPtr bufptr, ConvExec* ex) {
  std::string e = pack_weights_stream(cs, W, B, S, bf16, &pk);
  if (!e.empty()) return fail(ctx, SS4K_E_WEIGHTS, e);
  StreamParams& p = ex->sp;
  memset(&p, 0, sizeof(p));
  ex->stream = true;
  ex->nout = pk.nout;
  ex->name = cs.name;
  CK(ctx, cudaMalloc(&ex->d_w, pk.w.size() * 2));
  ex->w_bytes = pk.w.size() * 2;
  CK(ctx, cudaMemcpy(ex->d_w, pk.w.data(), pk.w.size() * 2, cudaMemcpyHostToDevice));
  CK(ctx, cudaMalloc(&ex->d_bias, pk.bias_f.size() * 4));
  CK(ctx, cudaMemcpy(ex->d_bias, pk.bias_f.data(), pk.bias_f.size() * 4, cudaMemcpyHostToDevice));
  CK(ctx, cudaMalloc(&ex->d_slope, pk.slope.size() * 4));
  CK(ctx, cudaMemcpy(ex->d_slope, pk.slope.data(), pk.slope.size() * 4, cudaMemcpyHostToDevice));
  const CUtensorMapDataType dt = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  {  // activations: (64 channels, W, channel block, H, N) starting at channel in_coff
    //              stride 2: the pixel-pair view (64 channels, W/2 pairs, block of the 2*pitch merged channels, H, N)
    const cuuint64_t eb = 2;
    const int avail = cs.in_pitch - cs.in_coff;
    const bool s2 = pk.stride2 != 0;
    const int nkb0 = s2 ? 2 * cs.in_pitch / 64 : (cs.cin + 63) / 64;  // 64-channel blocks of the source (split mode: 3 K blocks each)
    cuuint64_t dims[5] = {static_cast<cuuint64_t>(s2 ? 64 : (nkb0 == 1 ? std::min(64, avail) : 64)),
                          static_cast<cuuint64_t>(s2 ? cs.in_w / 2 : cs.in_w),
                          static_cast<cuuint64_t>(nkb0), static_cast<cuuint64_t>(cs.in_h),
                          static_cast<cuuint64_t>(cs.in_ring ? cs.in_ring : (cs.n_total > 0 ? cs.n_total : cs.n))};
    cuuint64_t strides[4] = {(s2 ? 2 : 1) * cs.in_pitch * eb, 128, static_cast<cuuint64_t>(cs.in_w) * cs.in_pitch * eb,
                             static_cast<cuuint64_t>(cs.in_h) * cs.in_w * cs.in_pitch * eb};
    cuuint32_t box[5] = {64, static_cast<cuuint32_t>(kBoxW), 1, 1, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    void* base = reinterpret_cast<uint8_t*>(bufptr(cs.in_buf)) + static_cast<size_t>(cs.in_coff) * 2;
    CUresult r = ctx->encode(&p.tmA[0], dt, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, SS4K_E_CUDA, fmt("cuTensorMapEncodeTiled(stream activation, %s) failed: %d", cs.name.c_str(), (int)r));
    p.tmA[1] = p.tmA[0];
    if (cs.split) {
      void* base_lo = reinterpret_cast<uint8_t*>(bufptr(cs.in_lo_buf)) + static_cast<size_t>(cs.in_coff) * 2;
      r = ctx->encode(&p.tmA[1], dt, 5, base_lo, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(ctx, SS4K_E_CUDA, fmt("cuTensorMapEncodeTiled(stream activation lo, %s) failed: %d", cs.name.c_str(), (int)r));
    }
  }
  {  // weights: rows of 64 channels
    const cuuint64_t rows = pk.w.size() / 64;
    cuuint64_t dims[2] = {64, rows};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(3 * pk.nout)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = ctx->encode(&p.tmW, dt, 2, ex->d_w, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, SS4K_E_CUDA, fmt("cuTensorMapEncodeTiled(stream weights) failed: %d", (int)r));
  }
  p.bias_f = ex->d_bias;
  p.bias_row0 = pk.bias_row0;
  p.tmB = p.tmW;
  if (stream_bias_mma(pk.nout)) {  // bias tiles: same tensor, NOUT-row box
    const cuuint64_t rows = pk.w.size() / 64;
    cuuint64_t dims[2] = {64, rows};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(pk.nout)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = ctx->encode(&p.tmB, dt, 2, ex->d_w, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, SS4K_E_CUDA, fmt("cuTensorMapEncodeTiled(stream bias) failed: %d", (int)r));
  }
  // fast epilogue: plain NHWC 16-bit output -> swizzled shared-memory tile -> TMA store
  p.fast_store = 0;
  p.stage_keep = getenv("SS4K_KEEP_STAGE") != nullptr ? 1u : 0u;
  if (stream_fast_store_ok(cs, pk.nout) && (cs.out_lo_buf < 0 || pk.split_fast)) {
    const cuuint64_t eb = 2;
    const int cavail = std::min(cs.out_pitch - cs.out_coff, pk.npad_total);
    const int out_imgs = cs.out_ring ? cs.out_ring : (cs.n_total > 0 ? cs.n_total : cs.n);
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(cavail), static_cast<cuuint64_t>(cs.out_w), static_cast<cuuint64_t>(cs.out_h),
                          static_cast<cuuint64_t>(out_imgs)};
    cuuint64_t strides[3] = {cs.out_pitch * eb, static_cast<cuuint64_t>(cs.out_w) * cs.out_pitch * eb,
                             static_cast<cuuint64_t>(cs.out_h) * cs.out_w * cs.out_pitch * eb};
    cuuint32_t box[4] = {static_cast<cuuint32_t>(pk.nout), 32, 1, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    const CUtensorMapSwizzle sw = pk.nout == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (pk.nout == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    void* base = reinterpret_cast<uint8_t*>(bufptr(cs.out_buf)) + static_cast<size_t>(cs.out_coff) * 2;
    CUresult r;
    if (cs.out_mode == kOutPS2NHWC) {
      // PixelShuffle(2) in the store: the shuffled tensor [N, 2H, 2W, pitch] viewed as (C, b, W, a, N*H); a chunk writes the
      // 32-pixel row segment of one sub-pixel phase (a, b)
      const cuuint64_t pb = cs.out_pitch * eb;
      const int cw = cs.in_w, chh = cs.in_h;   // conv resolution
      cuuint64_t d5[5] = {static_cast<cuuint64_t>(std::min(cs.out_pitch - cs.out_coff, cs.cout / 4)), 2, static_cast<cuuint64_t>(cw), 2,
                          static_cast<cuuint64_t>(chh) * out_imgs};
      cuuint64_t s5[4] = {pb, 2 * pb, 2 * static_cast<cuuint64_t>(cw) * pb, 4 * static_cast<cuuint64_t>(cw) * pb};
      cuuint32_t b5[5] = {static_cast<cuuint32_t>(pk.nout), 1, 32, 1, 1};
      r = ctx->encode(&p.tmO, dt, 5, base, d5, s5, b5, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r == CUDA_SUCCESS && pk.split_fast) {
        void* base_lo = reinterpret_cast<uint8_t*>(bufptr(cs.out_lo_buf)) + static_cast<size_t>(cs.out_coff) * 2;
        r = ctx->encode(&p.tmO2, dt, 5, base_lo, d5, s5, b5, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      }
      p.ps2 = 1;
    } else if (cs.up2_store) {
      // nearest-x2 upsample in the store: destination viewed as (C, b, W, a, N*H): pixel (2y+a, 2x+b) of the 2H x 2W image
      const cuuint64_t pb = cs.out_pitch * eb;
      cuuint64_t d5[5] = {static_cast<cuuint64_t>(cavail), 2, static_cast<cuuint64_t>(cs.out_w), 2,
                          static_cast<cuuint64_t>(cs.out_h) * out_imgs};
      cuuint64_t s5[4] = {pb, 2 * pb, 2 * static_cast<cuuint64_t>(cs.out_w) * pb, 4 * static_cast<cuuint64_t>(cs.out_w) * pb};
      cuuint32_t b5[5] = {static_cast<cuuint32_t>(pk.nout), 1, 32, 1, 1};
      r = ctx->encode(&p.tmO, dt, 5, base, d5, s5, b5, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
      r = ctx->encode(&p.tmO, dt, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                      CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r == CUDA_SUCCESS && pk.split_fast && cs.out_mode != kOutPS2NHWC) {
      void* base_lo = reinterpret_cast<uint8_t*>(bufptr(cs.out_lo_buf)) + static_cast<size_t>(cs.out_coff) * 2;
      r = ctx->encode(&p.tmO2, dt, 4, base_lo, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                      CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) return fail(ctx, SS4K_E_CUDA, fmt("cuTensorMapEncodeTiled(stream output, %s) failed: %d", cs.name.c_str(), (int)r));
    p.fast_store = pk.split_fast ? 3 : (cs.up2_store ? 2 : 1);
  }
  p.nkb = pk.nkb;
  for (int kb = 0; kb < pk.nkb; ++kb) { p.a_kb[kb] = pk.src_kb[kb]; p.a_tm[kb] = pk.src_tm[kb]; p.nks[kb] = pk.nks[kb]; p.wt[kb] = pk.wt[kb]; }
  p.nwt = pk.nwt;
  p.n_in0 = cs.n0; p.n_out0 = cs.n0;   // TMA image coordinates of a step that starts inside the clip
  p.ring_in = p.ring_out = p.ring_res1 = p.ring_res2 = -1;   // no ring wrap (BSVD streams set theirs per tensor)
  p.stride2 = pk.stride2; p.nkx = pk.nkx;
  for (int kb = 0; kb < pk.nkb; ++kb) { p.ksm[kb][0] = pk.ksm[kb][0]; p.ksm[kb][1] = pk.ksm[kb][1]; }
  p.n_img = cs.n; p.H = pk.stride2 ? cs.in_h / 2 : cs.in_h; p.W = pk.stride2 ? cs.in_w / 2 : cs.in_w;  // the output grid
  p.strips = (p.W + kTileW - 1) / kTileW;
  p.chunks = pk.chunks;
  p.total_units = pk.chunks * cs.n * p.strips * p.H;
  p.acc_slots = pk.acc_slots; p.a_slots = pk.a_slots;
  p.l2_in = cs.l2_in; p.l2_out = cs.l2_out;
  if (const char* e = getenv("SS4K_DBG_FLAGS")) {  // experiments only (see StreamParams::dbg_flags): RRDB trunk convs
    if (cs.name.rfind("body.", 0) == 0) p.dbg_flags = atoi(e);
  }
  if (cs.discard_buf >= 0 && cs.discard_mask != 0) {
    p.discard_ptr = bufptr(cs.discard_buf);
    p.discard_pitch_bytes = static_cast<uint32_t>(cs.discard_pitch) * 2u;
    p.discard_mask = static_cast<uint32_t>(cs.discard_mask);
    p.discard_npx = cs.discard_npx;
  }
  const uint32_t f = bf16 ? 1u : 0u;
  for (int i = 0; i < 3; ++i)
    p.idesc[i] = (1u << 4) | (f << 7) | (f << 10) | (static_cast<uint32_t>((i + 1) * pk.nout >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
  p.err = ctx->err_dev;
  fill_epilogue(cs, bf16, bufptr, ex->d_bias, ex->d_slope, &p.ep, &ex->ext_out);
  p.ep.bias = nullptr;                  // the accumulators start from the bias (p.bias_f)
  p.ep.slope = S ? ex->d_slope : nullptr;
  p.ep.slope_const = cs.const_slope;
  p.ep.alpha = pk.alpha_out;            // folded into weights / bias when the activation allows
  ex->grid = std::min(p.total_units, ctx->nsm);
  return SS4K_OK;
}

const bool g_use_pdl = getenv("SS4K_NO_PDL") == nullptr;

cudaError_t launch_exec(const ConvExec& c, void* ext_out, cudaStream_t st) {
  if (c.stream) {
    if (c.ext_out) {
      StreamParams p = c.sp;
      p.ep.out = ext_out;
      return conv_stream_launch(p, c.nout, c.grid, st, g_use_pdl);
    }
    return conv_stream_launch(c.sp, c.nout, c.grid, st, g_use_pdl);
  }
  if (c.ext_out) {
    ConvParams p = c.p;
    p.ep.out = ext_out;
    return conv_tc_launch(p, c.grid, st);
  }
  return conv_tc_launch(c.p, c.grid, st);
}

// Build the kernel parameter block of one conv.  bufptr(id) resolves program buffer ids.
template <class BufPtr>
int materialize_conv(ss4k_ctx* ctx, const ConvSpec& cs, const HostTensor& W, const HostTensor* B,
                     const HostTensor* S, int act_mode, BufPtr bufptr, ConvExec* ex) {
  const bool bf16 = act_mode == SS4K_ACT_BF16;
  {
    StreamPacked spk;
    if (stream_config(cs, &spk)) return materialize_stream(ctx, cs, W, B, S, bf16, spk, bufptr, ex);
  }
  PackedWeights pw;
  std::string e = pack_weights(cs, W, B, S, bf16, &pw);
  if (!e.empty()) return fail(ctx, SS4K_E_WEIGHTS, e);
  ConvParams& p = ex->p;
  memset(&p, 0, sizeof(p));
  ex->name = cs.name;
  // A-space geometry
  int AH = cs.in_h, AW = cs.in_w;
  if (cs.mode == kModeS2) { AH = cs.in_h / 2; AW = cs.in_w / 2; }
  TileCfg t;
  e = configure_tiles(ctx->desc_mode, ctx->nsm, cs.n, AH, AW, pw.npad_total, pw.ntaps, pw.nsub, pw.max_dr, pw.nkb, &t);
  if (!e.empty()) return fail(ctx, SS4K_E_INVALID, "conv " + cs.name + ": " + e);
  // upload weights
  CK(ctx, cudaMalloc(&ex->d_w, pw.w.size() * 2));
  CK(ctx, cudaMemcpy(ex->d_w, pw.w.data(), pw.w.size() * 2, cudaMemcpyHostToDevice));
  CK(ctx, cudaMalloc(&ex->d_bias, pw.bias.size() * 4));
  CK(ctx, cudaMemcpy(ex->d_bias, pw.bias.data(), pw.bias.size() * 4, cudaMemcpyHostToDevice));
  CK(ctx, cudaMalloc(&ex->d_slope, pw.slope.size() * 4));
  CK(ctx, cudaMemcpy(ex->d_slope, pw.slope.data(), pw.slope.size() * 4, cudaMemcpyHostToDevice));
  // tensor maps
  const int box_w = ctx->desc_mode == 2 ? kTileW : kBoxW;
  const int in_imgs = cs.in_ring ? cs.in_ring : (cs.n_total > 0 ? cs.n_total : cs.n);
  e = encode_act_map(ctx, &p.tmA[0], bufptr(cs.in_buf), in_imgs, cs.in_h, cs.in_w, cs.in_pitch, cs.mode, bf16, box_w);
  if (!e.empty()) return fail(ctx, SS4K_E_CUDA, e);
  if (cs.split) {
    e = encode_act_map(ctx, &p.tmA[1], bufptr(cs.in_lo_buf), in_imgs, cs.in_h, cs.in_w, cs.in_pitch, cs.mode, bf16, box_w);
    if (!e.empty()) return fail(ctx, SS4K_E_CUDA, e);
  } else {
    p.tmA[1] = p.tmA[0];
  }
  e = encode_w_map(ctx, &p.tmW, ex->d_w, pw.npad_total, pw.nkb * pw.ntaps, t.n_cta, pw.ntaps, bf16);
  if (!e.empty()) return fail(ctx, SS4K_E_CUDA, e);
  // schedule tables
  p.nkb = pw.nkb; p.ntaps = pw.ntaps; p.nsub = pw.nsub; p.max_dr = pw.max_dr; p.mode = cs.mode;
  for (int i = 0; i < pw.nkb; ++i) p.kb[i] = pw.kb[i];
  for (int i = 0; i < pw.ntaps; ++i) p.taps[i] = pw.taps[i];
  for (int i = 0; i < pw.nkb; ++i)
    for (int j = 0; j < kMaxTaps; ++j) p.ksmask[i][j] = pw.mask[static_cast<size_t>(i) * kMaxTaps + j];
  p.n_img = cs.n; p.H = AH; p.W = AW; p.R = t.R;
  p.n_in0 = cs.n0;
  p.tiles_x = t.tiles_x; p.tiles_y = t.tiles_y; p.n_chunks = t.n_chunks; p.n_tiles = t.n_tiles;
  p.n_cta = t.n_cta; p.acc_stride = t.acc_stride;
  p.a_slots = t.a_slots; p.a_slot_bytes = t.a_slot_bytes; p.a_sub_bytes = t.a_sub_bytes;
  p.w_slots = t.w_slots; p.w_slot_bytes = t.w_slot_bytes; p.w_tile_bytes = t.w_tile_bytes;
  p.w_resident = t.w_resident;
  p.desc_mode = ctx->desc_mode;
  const uint32_t f = bf16 ? 1u : 0u;
  p.idesc = (1u << 4) | (f << 7) | (f << 10) | (static_cast<uint32_t>(t.n_cta >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
  p.a_row_tx = ctx->desc_mode == 2 ? 3u * kTileW * kRowBytes : static_cast<uint32_t>(kBoxW) * kRowBytes;
  p.w_tx = static_cast<uint32_t>(t.w_slot_bytes);
  p.err = ctx->err_dev;
  fill_epilogue(cs, bf16, bufptr, ex->d_bias, ex->d_slope, &p.ep, &ex->ext_out);
  ex->grid = std::min(t.n_tiles, ctx->nsm);
  return SS4K_OK;
}

int check_kernel_health(ss4k_ctx* ctx, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return SS4K_OK;
  std::string msg = fmt("%s: %s", what, cudaGetErrorString(e));
  if (ctx && ctx->err_host && ctx->err_host[0] != 0)
    msg += fmt(" [pipeline watchdog: wait tag %d block %d thread %d parity %d]", ctx->err_host[0], ctx->err_host[1],
               ctx->err_host[2], ctx->err_host[3]);
  return fail(ctx, SS4K_E_CUDA, msg);
}

}  // namespace

// ================================================================================================
struct ss4k_plan {
  ss4k_ctx* ctx = nullptr;
  ss4k_plan_cfg cfg;
  Program prog;
  std::vector<void*> bufs;
  std::vector<ConvExec> convs;  // one per conv step, in step order
  std::vector<int> step_conv;   // step index -> conv index (or -1)
  cudaGraphExec_t graph = nullptr;
  int graph_first = -1, graph_last = -1;  // [first, last] step range inside the graph
  int fused_prep = -1;   // step index of a layout (prep) step whose work the following conv's loader does, or -1
  int32_t* d_mask = nullptr;  // masked canvases (cfg.reserved[5]): crop size (h, w) of every image of the batch at the input resolution
  void* stage_in = nullptr;   // device staging for ss4k_run_host
  void* stage_out = nullptr;
  // NV12 output in two steps (tiled plans, or a last conv that does not run on the streaming kernel): the uint8 RGB frame
  // the last conv / the tile paste writes, converted into the caller's buffer by the rgb_to_nv12 kernel.  Null when the
  // last conv's epilogue stores NV12 itself.
  void* nv12_rgb = nullptr;
  // software pipeline of ss4k_run_host_async: two staging slots, copy streams, hand-over events
  struct HostPipe {
    void* in[2] = {nullptr, nullptr};
    void* out[2] = {nullptr, nullptr};
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t in_ready[2] = {nullptr, nullptr}, out_ready[2] = {nullptr, nullptr}, out_copied[2] = {nullptr, nullptr};
    uint64_t calls = 0;
    bool init = false;
  } pipe;
  int64_t in_bytes = 0, out_bytes = 0;
  // tiled inference (cfg.tile / tile_pad / pre_pad, RealESRGANer semantics): one sub-plan per padded-crop shape class
  struct TileClass {
    int hc = 0, wc = 0, count = 0;   // canvas of the group's atlas images, number of crops
    int nimg = 1;                    // atlas images per frame
    ss4k_plan* sub = nullptr;
    TileBox* d_boxes = nullptr;
    void* d_in = nullptr;
    void* d_out = nullptr;
  };
  std::vector<TileClass> tiles;
  bool tiled = false;
};

namespace {

int64_t fmt_bytes(int fmtid, int n, int c, int h, int w) {
  switch (fmtid) {
    case SS4K_FMT_F32_NCHW: return static_cast<int64_t>(n) * c * h * w * 4;
    case SS4K_FMT_F16_NCHW: return static_cast<int64_t>(n) * c * h * w * 2;
    case SS4K_FMT_U8_NHWC: return static_cast<int64_t>(n) * c * h * w;
    case SS4K_FMT_NV12: return static_cast<int64_t>(n) * h * w * 3 / 2;
    default: return 0;
  }
}

int run_step(ss4k_plan* pl, int si, const void* in_dev, void* out_dev, cudaStream_t st) {
  ss4k_ctx* ctx = pl->ctx;
  const Step& s = pl->prog.steps[si];
  if (s.kind == 0) {
    if (si == pl->fused_prep) return SS4K_OK;   // decoded by the first conv's producer warp (StreamParams::src)
    const PrepSpec& p = s.prep;
    const bool bf16 = pl->cfg.act_mode == SS4K_ACT_BF16;
    // (a BSVD chunk with a temporal halo converts only the frames [n0, n0 + n) the owned outputs depend on)
    const BufSpec& ob = pl->prog.bufs[p.out_buf];
    const size_t in_off = static_cast<size_t>(fmt_bytes(p.in_fmt, 1, pl->prog.in_c, p.h, p.w)) * p.n0;
    const size_t out_off = static_cast<size_t>(ob.h) * ob.w * ob.pitch * 2 * p.n0;
    CK(ctx, prep_launch(p.in_fmt, reinterpret_cast<const uint8_t*>(in_dev) + in_off, reinterpret_cast<uint8_t*>(pl->bufs[p.out_buf]) + out_off,
                        p.out_lo_buf >= 0 ? reinterpret_cast<uint8_t*>(pl->bufs[p.out_lo_buf]) + out_off : nullptr,
                        p.n, p.c, p.h, p.w, ob.pitch, p.unshuffle, p.fill_ch, p.fill_val, bf16 ? 1 : 0, st));
    ctx->launches++;
  } else if (s.kind == 2) {
    const Program& P = pl->prog;
    CK(ctx, rgb_to_nv12_launch(pl->nv12_rgb, out_dev, P.out_n, P.out_h, P.out_w, st));
    ctx->launches++;
  } else {
    ConvExec& c = pl->convs[pl->step_conv[si]];
    if (c.src_ext) c.sp.src = reinterpret_cast<const uint8_t*>(in_dev) + c.src_off;
    // (two-step NV12 output: the last conv writes the plan's uint8 RGB frame, the conversion step the caller's buffer)
    CK(ctx, launch_exec(c, c.ext_out && pl->nv12_rgb != nullptr ? pl->nv12_rgb : out_dev, st));
    ctx->launches++;
  }
  return SS4K_OK;
}

bool step_is_external(const Step& s) {
  if (s.kind != 1) return true;  // prep reads the caller's pointer, the NV12 conversion writes it
  return s.conv.out_buf == kBufExternalOut;
}

// North-star part 4 (colour conversion in the first layer's load): a BSVD clip plan fed with uint8 RGB / NV12 frames
// does not run its layout step; the first conv's producer warp decodes the frames into its activation slabs and leaves
// the 16-bit rows for the DenBlock's residual (StreamParams::src).  Streaming convs of the <32> kernel only.
void fuse_prep(ss4k_plan* pl) {
  Program& P = pl->prog;
  if (getenv("SS4K_NO_FUSED_PREP") != nullptr || P.steps.size() < 2 || pl->cfg.arch != SS4K_ARCH_BSVD) return;
  const Step& s0 = P.steps[0];
  const Step& s1 = P.steps[1];
  if (s0.kind != 0 || s1.kind != 1) return;
  const PrepSpec& pp = s0.prep;
  const ConvSpec& cs = s1.conv;
  if ((pp.in_fmt != SS4K_FMT_U8_NHWC && pp.in_fmt != SS4K_FMT_NV12) || pp.unshuffle != 1 || pp.c != 3) return;
  if (pp.w % 4 != 0) return;   // the decoder warps read four pixels with aligned 32-bit loads
  if (cs.in_buf != pp.out_buf || cs.mode != kModeConv3 || cs.in_pitch != 16 || cs.in_coff != 0 || cs.cin > 8) return;
  if (pl->cfg.act_mode == SS4K_ACT_BF16) return;
  if (pp.fill_ch >= 0 && pp.fill_ch != 3) return;
  ConvExec& c = pl->convs[pl->step_conv[1]];
  if (!c.stream) return;
  // the conv must cover every frame the layout step would have converted for other readers (the residual of the block's
  // last conv): its frame range contains theirs by construction (bsvd_program.cpp), check it anyway
  const int c0 = cs.n0, c1 = cs.n0 + cs.n;
  for (size_t si = 2; si < P.steps.size(); ++si) {
    if (P.steps[si].kind != 1) continue;
    const ConvSpec& o = P.steps[si].conv;
    const bool reads = o.in_buf == pp.out_buf || o.res1_buf == pp.out_buf || o.res2_buf == pp.out_buf;
    if (reads && (o.n0 < c0 || o.n0 + o.n > c1)) return;
  }
  StreamParams& sp = c.sp;
  sp.src_fmt = pp.in_fmt;
  sp.src_fill_ch = pp.fill_ch;
  sp.src_fill = pp.fill_val;
  sp.src_out = reinterpret_cast<uint16_t*>(pl->bufs[pp.out_buf]);
  sp.src_out_lo = pp.out_lo_buf >= 0 ? reinterpret_cast<uint16_t*>(pl->bufs[pp.out_lo_buf]) : nullptr;
  c.src_ext = true;
  c.src_off = 0;   // (sp.n_in0 carries the step's first frame)
  pl->fused_prep = 0;
}

}  // namespace

extern "C" {

int ss4k_abi_version(void) { return SS4K_ABI_VERSION; }

const char* ss4k_last_error(ss4k_ctx* ctx) {
  if (ctx) return ctx->err.c_str();
  return g_last_error.c_str();
}

void ss4k_free(void* p) { free(p); }

static int self_probe(ss4k_ctx* ctx);

int ss4k_create(int device_id, ss4k_ctx** out_ctx) {
  if (!out_ctx) return fail(nullptr, SS4K_E_INVALID, "out_ctx is null");
  *out_ctx = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, SS4K_E_NODEVICE,
                fmt("no CUDA device (%s); this engine has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e)));
  if (device_id < 0 || device_id >= ndev) return fail(nullptr, SS4K_E_INVALID, "device_id out of range");
  cudaDeviceProp prop;
  CK(nullptr, cudaGetDeviceProperties(&prop, device_id));
  if (prop.major != 10)
    return fail(nullptr, SS4K_E_NODEVICE, fmt("device %d is sm_%d%d; this engine is written for sm_100a (B200)", device_id, prop.major, prop.minor));
  CK(nullptr, cudaSetDevice(device_id));
  std::unique_ptr<ss4k_ctx> ctx(new ss4k_ctx());
  ctx->device = device_id;
  ctx->nsm = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CK(nullptr, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(nullptr, SS4K_E_NODEVICE, "cuTensorMapEncodeTiled not available in this driver");
  ctx->encode = reinterpret_cast<EncodeTiledFn>(fn);
  CK(nullptr, cudaHostAlloc(reinterpret_cast<void**>(&ctx->err_host), 16, cudaHostAllocMapped));
  memset(ctx->err_host, 0, 16);
  CK(nullptr, cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->err_dev), ctx->err_host, 0));
  CK(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CK(nullptr, conv_tc_prepare());
  CK(nullptr, conv_stream_prepare());
  const char* force = getenv("SS4K_DESC_MODE");
  if (force && *force) {
    ctx->desc_mode = atoi(force);
    if (getenv("SS4K_SKIP_PROBE") == nullptr) {
      int rc = self_probe(ctx.get());
      if (rc != SS4K_OK) { g_last_error = ctx->err; return rc; }
    }
  } else {
    int rc = SS4K_E_SELFTEST;
    std::string log;
    for (int mode = 0; mode < 3; ++mode) {
      ctx->desc_mode = mode;
      rc = self_probe(ctx.get());
      if (rc == SS4K_OK) break;
      log += fmt("[mode %d: %s] ", mode, ctx->err.c_str());
      if (rc != SS4K_E_SELFTEST) break;  // CUDA error: context is likely poisoned
    }
    if (rc != SS4K_OK) return fail(nullptr, rc, "tcgen05 self-probe failed: " + log);
  }
  *out_ctx = ctx.release();
  return SS4K_OK;
}

int ss4k_destroy(ss4k_ctx* ctx) {
  if (!ctx) return SS4K_OK;
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->err_host) cudaFreeHost(ctx->err_host);
  delete ctx;
  return SS4K_OK;
}

int ss4k_desc_mode(ss4k_ctx* ctx) { return ctx ? ctx->desc_mode : -1; }
int ss4k_set_desc_mode(ss4k_ctx* ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return fail(ctx, SS4K_E_INVALID, "bad desc mode");
  ctx->desc_mode = mode;
  return SS4K_OK;
}
int64_t ss4k_launch_count(ss4k_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ss4k_load_weights(ss4k_ctx* ctx, int net_id, const char* name, const void* host_ptr, int dtype,
                      const int64_t* shape, int ndim) {
  if (!ctx || !name || !host_ptr || !shape || ndim < 1 || ndim > 4) return fail(ctx, SS4K_E_INVALID, "bad argument to ss4k_load_weights");
  HostTensor t;
  size_t count = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); count *= static_cast<size_t>(shape[i]); }
  t.data.resize(count);
  if (dtype == SS4K_DT_F32) {
    memcpy(t.data.data(), host_ptr, count * 4);
  } else if (dtype == SS4K_DT_F16) {
    const uint16_t* h = reinterpret_cast<const uint16_t*>(host_ptr);
    for (size_t i = 0; i < count; ++i) t.data[i] = h2f(h[i], false);
  } else {
    return fail(ctx, SS4K_E_INVALID, "unsupported weight dtype");
  }
  ctx->weights[net_id][name] = std::move(t);
  return SS4K_OK;
}

int ss4k_clear_weights(ss4k_ctx* ctx, int net_id) {
  if (!ctx) return SS4K_E_INVALID;
  ctx->weights.erase(net_id);
  return SS4K_OK;
}

static PlanCfgLite lite(const ss4k_plan_cfg* c) {
  PlanCfgLite l;
  l.arch = c->arch; l.n = c->n; l.h = c->h; l.w = c->w; l.scale = c->scale; l.depth = c->depth;
  l.tile = c->tile; l.tile_pad = c->tile_pad; l.act_mode = c->act_mode; l.in_fmt = c->in_fmt; l.out_fmt = c->out_fmt;
  memcpy(&l.bsvd_noise, &c->reserved[0], 4);
  l.own_lo = c->reserved[2]; l.own_hi = c->reserved[3];
  return l;
}

int ss4k_plan_dry(const ss4k_plan_cfg* cfg, char** out_json) {
  if (!cfg || !out_json) return fail(nullptr, SS4K_E_INVALID, "null argument");
  Program prog;
  std::string e = build_program(lite(cfg), &prog);
  if (!e.empty()) return fail(nullptr, SS4K_E_INVALID, e);
  std::string js = prog.to_json();
  *out_json = static_cast<char*>(malloc(js.size() + 1));
  memcpy(*out_json, js.c_str(), js.size() + 1);
  return SS4K_OK;
}

int ss4k_plan_destroy(ss4k_plan* pl) {
  if (!pl) return SS4K_OK;
  for (auto& t : pl->tiles) {
    if (t.sub) ss4k_plan_destroy(t.sub);
    if (t.d_boxes) cudaFree(t.d_boxes);
    if (t.d_in) cudaFree(t.d_in);
    if (t.d_out) cudaFree(t.d_out);
  }
  if (pl->graph) cudaGraphExecDestroy(pl->graph);
  for (auto& c : pl->convs) free_conv(c);
  for (void* b : pl->bufs) if (b) cudaFree(b);
  if (pl->pipe.init) {
    cudaStreamSynchronize(pl->pipe.h2d);
    cudaStreamSynchronize(pl->pipe.d2h);
    for (int i = 0; i < 2; ++i) {
      cudaFree(pl->pipe.in[i]); cudaFree(pl->pipe.out[i]);
      cudaEventDestroy(pl->pipe.in_ready[i]); cudaEventDestroy(pl->pipe.out_ready[i]); cudaEventDestroy(pl->pipe.out_copied[i]);
    }
    cudaStreamDestroy(pl->pipe.h2d); cudaStreamDestroy(pl->pipe.d2h);
  }
  if (pl->stage_in) cudaFree(pl->stage_in);
  if (pl->stage_out) cudaFree(pl->stage_out);
  if (pl->nv12_rgb) cudaFree(pl->nv12_rgb);
  if (pl->d_mask) cudaFree(pl->d_mask);
  delete pl;
  return SS4K_OK;
}

static int create_tiled_plan(ss4k_ctx* ctx, const ss4k_plan_cfg* cfg, ss4k_plan** out_plan);

int ss4k_plan_create(ss4k_ctx* ctx, const ss4k_plan_cfg* cfg, ss4k_plan** out_plan) {
  if (!ctx || !cfg || !out_plan) return fail(ctx, SS4K_E_INVALID, "null argument");
  *out_plan = nullptr;
  DeviceGuard dev_guard(ctx->device);
  if (cfg->arch != SS4K_ARCH_BSVD) {
    // RealESRGANer options (factory.py:93-95): tile / tile_pad / pre_pad, and the reflect mod-pad of the x2 nets
    const int pre_pad = cfg->reserved[1];
    const bool mod2 = cfg->arch == SS4K_ARCH_RRDB && cfg->scale == 2 && (((cfg->h + pre_pad) | (cfg->w + pre_pad)) & 1);
    const bool one_tile = cfg->tile > 0 && cfg->tile >= cfg->h && cfg->tile >= cfg->w;   // a single tile is the frame itself
    if (pre_pad < 0 || cfg->tile < 0 || cfg->tile_pad < 0) return fail(ctx, SS4K_E_INVALID, "negative tile / tile_pad / pre_pad");
    if ((cfg->tile > 0 && !one_tile) || pre_pad > 0 || mod2) return create_tiled_plan(ctx, cfg, out_plan);
  }
  std::unique_ptr<ss4k_plan> pl(new ss4k_plan());
  pl->ctx = ctx;
  pl->cfg = *cfg;
  std::string e = build_program(lite(cfg), &pl->prog);
  if (!e.empty()) return fail(ctx, SS4K_E_INVALID, e);
  auto wit = ctx->weights.find(cfg->net_id);
  if (wit == ctx->weights.end()) return fail(ctx, SS4K_E_WEIGHTS, fmt("no weights loaded for net_id %d", cfg->net_id));
  const auto& wmap = wit->second;
  Program& P = pl->prog;
  // buffers
  pl->bufs.assign(P.bufs.size(), nullptr);
  for (size_t i = 0; i < P.bufs.size(); ++i) {
    cudaError_t ce = cudaMalloc(&pl->bufs[i], P.bufs[i].bytes());
    if (ce != cudaSuccess) {
      int rc = fail(ctx, SS4K_E_NOMEM, fmt("cudaMalloc(%zu bytes) for buffer %s failed: %s", P.bufs[i].bytes(), P.bufs[i].name.c_str(), cudaGetErrorString(ce)));
      ss4k_plan_destroy(pl.release());
      return rc;
    }
    cudaMemset(pl->bufs[i], 0, P.bufs[i].bytes());
  }
  auto bufptr = [&](int id) -> void* { return id >= 0 ? pl->bufs[id] : nullptr; };
  // convs
  pl->step_conv.assign(P.steps.size(), -1);
  pl->convs.reserve(P.steps.size());
  bool nv12_two_step = false;
  for (size_t si = 0; si < P.steps.size(); ++si) {
    if (P.steps[si].kind != 1) continue;
    if (P.steps[si].conv.out_mode == kOutNV12 && !stream_nv12_ok(P.steps[si].conv)) {
      P.steps[si].conv.out_mode = kOutU8NHWC;   // two-step form: uint8 RGB into pl->nv12_rgb, then the conversion step
      nv12_two_step = true;
    }
    const ConvSpec& cs = P.steps[si].conv;
    auto w = wmap.find(cs.wname);
    if (w == wmap.end()) { int rc = fail(ctx, SS4K_E_WEIGHTS, "missing weight " + cs.wname); ss4k_plan_destroy(pl.release()); return rc; }
    const HostTensor* B = nullptr;
    const HostTensor* S = nullptr;
    if (!cs.bname.empty()) {
      auto b = wmap.find(cs.bname);
      if (b == wmap.end()) { int rc = fail(ctx, SS4K_E_WEIGHTS, "missing bias " + cs.bname); ss4k_plan_destroy(pl.release()); return rc; }
      B = &b->second;
    }
    if (!cs.sname.empty()) {
      auto s = wmap.find(cs.sname);
      if (s == wmap.end()) { int rc = fail(ctx, SS4K_E_WEIGHTS, "missing PReLU slope " + cs.sname); ss4k_plan_destroy(pl.release()); return rc; }
      S = &s->second;
    }
    pl->convs.emplace_back();
    pl->step_conv[si] = static_cast<int>(pl->convs.size()) - 1;
    int rc = materialize_conv(ctx, cs, w->second, B, S, cfg->act_mode, bufptr, &pl->convs.back());
    if (rc != SS4K_OK) { ss4k_plan_destroy(pl.release()); return rc; }
  }
  if (nv12_two_step) {
    cudaError_t ce = cudaMalloc(&pl->nv12_rgb, fmt_bytes(SS4K_FMT_U8_NHWC, P.out_n, 3, P.out_h, P.out_w) + 256);
    if (ce != cudaSuccess) { ss4k_plan_destroy(pl.release()); return fail(ctx, SS4K_E_NOMEM, "NV12 output: uint8 RGB frame"); }
    Step s;
    s.kind = 2;
    P.steps.push_back(s);
    pl->step_conv.push_back(-1);
  }
  fuse_prep(pl.get());
  if (cfg->reserved[5] == 1) {
    // masked canvases (tiled inference): every conv zeroes its output outside the image's crop; needs every conv on the
    // streaming kernel, at a power-of-two multiple of the input resolution
    std::vector<int32_t> hw(static_cast<size_t>(kMaskStride) * P.in_n, 0);
    for (int i = 0; i < P.in_n; ++i) {   // default: one crop = the whole canvas (the tiled plan fills in its atlases)
      int32_t* e = hw.data() + static_cast<size_t>(i) * kMaskStride;
      e[0] = 1; e[1] = 0; e[2] = P.in_w; e[3] = P.in_h;
    }
    cudaError_t ce = cudaMalloc(&pl->d_mask, hw.size() * sizeof(int32_t));
    if (ce == cudaSuccess) ce = cudaMemcpy(pl->d_mask, hw.data(), hw.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) { ss4k_plan_destroy(pl.release()); return fail(ctx, SS4K_E_NOMEM, "mask table"); }
    for (size_t si = 0; si < P.steps.size(); ++si) {
      if (P.steps[si].kind != 1) continue;
      const ConvSpec& cs = P.steps[si].conv;
      ConvExec& c = pl->convs[pl->step_conv[si]];
      int shift = 0, hh = P.in_h;
      bool ok = c.stream && cs.mode == kModeConv3 && cs.n == P.in_n;
      if (ok) {
        while (hh < cs.in_h && shift < 4) { hh *= 2; ++shift; }
        while (hh > cs.in_h && shift > -4) { if (hh & 1) { ok = false; break; } hh /= 2; --shift; }
        ok = ok && hh == cs.in_h &&
             (shift >= 0 ? (P.in_w << shift) == cs.in_w : (P.in_w >> -shift) == cs.in_w && (P.in_w & ((1 << -shift) - 1)) == 0);
      }
      if (!ok) { ss4k_plan_destroy(pl.release()); return fail(ctx, SS4K_E_INVALID, "masked canvases: conv " + cs.name + " is not a streaming conv at a power-of-two multiple of the input size"); }
      c.sp.mask_hw = pl->d_mask;
      c.sp.mask_shift = shift;
    }
  }
  // Early activation loads (StreamParams::early_kb_mask): K blocks that only read channels written at least two steps
  // ago are requested before the dependency wait.  Needs this conv and the two launches before it to be streaming convs
  // that fill every SM (see conv_params.h).
  if (getenv("SS4K_NO_EARLY_LOAD") == nullptr) {
    for (size_t si = 2; si < P.steps.size(); ++si) {
      if (P.steps[si].kind != 1 || P.steps[si - 1].kind != 1 || P.steps[si - 2].kind != 1) continue;
      ConvExec& c = pl->convs[pl->step_conv[si]];
      const ConvExec& p1 = pl->convs[pl->step_conv[si - 1]];
      const ConvExec& p2 = pl->convs[pl->step_conv[si - 2]];
      const ConvSpec& cs = P.steps[si].conv;
      if (!c.stream || !p1.stream || !p2.stream || c.grid != ctx->nsm || p1.grid != ctx->nsm || p2.grid != ctx->nsm) continue;
      if (cs.old_cin <= 0 || cs.split) continue;
      // the argument above needs exactly one resident CTA per SM
      if (conv_stream_max_ctas_per_sm(c.nout) != 1) continue;
      uint32_t mask = 0;
      for (int kb = 0; kb < c.sp.nkb; ++kb)
        if (c.sp.a_tm[kb] == 0 && (c.sp.a_kb[kb] + 1) * 64 <= cs.old_cin) mask |= 1u << kb;
      c.sp.early_kb_mask = mask;
    }
  }
  // each launch prefetches the next launch's packed weights into L2 (the last one: the first conv's, for the next frame)
  if (getenv("SS4K_NO_W_PREFETCH") == nullptr) {
    const int nc = static_cast<int>(pl->convs.size());
    for (int i = 0; i < nc; ++i) {
      ConvExec& c = pl->convs[i];
      const ConvExec& nx = pl->convs[(i + 1) % nc];
      if (nc < 2 || !c.stream || nx.d_w == nullptr || !nx.stream) continue;
      c.sp.next_w = nx.d_w; c.sp.next_w_bytes = static_cast<uint32_t>(nx.w_bytes);
    }
  }
  pl->in_bytes = fmt_bytes(P.in_fmt, P.in_n, P.in_c, P.in_h, P.in_w);
  pl->out_bytes = fmt_bytes(P.out_fmt, P.out_n, P.out_c, P.out_h, P.out_w);
  // CUDA graph over the internal (non-external) middle of the program
  if (cfg->use_graph) {
    int first = -1, last = -1;
    auto external = [&](size_t si) {
      return step_is_external(P.steps[si]) || (P.steps[si].kind == 1 && pl->convs[pl->step_conv[si]].src_ext);
    };
    for (size_t si = 0; si < P.steps.size(); ++si) {
      if (!external(si)) { if (first < 0) first = (int)si; last = (int)si; }
    }
    bool contiguous = first >= 0;
    for (int si = first; contiguous && si <= last; ++si) if (external(si)) contiguous = false;
    if (contiguous && last - first >= 1) {
      cudaGraph_t g = nullptr;
      int64_t saved = ctx->launches;
      cudaError_t ce = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
      int rc = SS4K_OK;
      if (ce == cudaSuccess) {
        for (int si = first; si <= last && rc == SS4K_OK; ++si) rc = run_step(pl.get(), si, nullptr, nullptr, ctx->stream);
        ce = cudaStreamEndCapture(ctx->stream, &g);
      }
      ctx->launches = saved;
      if (ce == cudaSuccess && rc == SS4K_OK && g) {
        ce = cudaGraphInstantiate(&pl->graph, g, 0);
        if (ce == cudaSuccess) { pl->graph_first = first; pl->graph_last = last; }
        else pl->graph = nullptr;
      }
      if (g) cudaGraphDestroy(g);
      cudaGetLastError();
    }
  }
  // weight uploads (pageable cudaMemcpy) and buffer memsets ran on the NULL stream; the plan runs on the caller's stream
  { cudaError_t ce = cudaDeviceSynchronize(); if (ce != cudaSuccess) { int rc = check_kernel_health(ctx, ce, "ss4k_plan_create"); ss4k_plan_destroy(pl.release()); return rc; } }
  *out_plan = pl.release();
  return SS4K_OK;
}

// ------------------------------------------------------------------------------------------------
// Tiled plans: RealESRGANer.pre_process (reflect pre_pad, mod-2 pad of the x2 nets), tile_process (grid of
// ceil(W/tile) x ceil(H/tile) tiles, each crop expanded by tile_pad and clamped to the padded frame, un-padded centre
// pasted, no blending) and post_process (pads cropped off) -- SURVEY.md Appendix B; reached from
// realesrgan/factory.py:93-95,160-169.  Crops of one shape are independent images: they run as ONE batch per class.
struct TileGroup { int hc = 0, wc = 0, nimg = 1; std::vector<TileBox> boxes; };

// Host-only: RealESRGANer's tile grid for a frame and its packing into crop atlases (see create_tiled_plan).
static std::string layout_tiles(const ss4k_plan_cfg* cfg, std::vector<TileGroup>* out_groups) {
  std::vector<TileGroup>& groups = *out_groups;
  groups.clear();
  if (cfg->in_fmt == SS4K_FMT_NV12) return "tiled inference takes RGB frames (float / half NCHW or uint8 NHWC)";
  const int s = cfg->scale;
  const int pre_pad = cfg->reserved[1];
  int Hp = cfg->h + pre_pad, Wp = cfg->w + pre_pad;
  if (cfg->arch == SS4K_ARCH_RRDB && s == 2) { Hp += Hp & 1; Wp += Wp & 1; }
  if (Hp - cfg->h >= cfg->h || Wp - cfg->w >= cfg->w) return "pre_pad must be smaller than the frame (reflect padding)";
  const int tile = cfg->tile > 0 ? cfg->tile : std::max(Hp, Wp);
  const int pad = cfg->tile > 0 ? cfg->tile_pad : 0;
  std::map<std::pair<int, int>, std::vector<TileBox>> classes;
  const int tx = (Wp + tile - 1) / tile, ty = (Hp + tile - 1) / tile;
  for (int y = 0; y < ty; ++y)
    for (int x = 0; x < tx; ++x) {
      const int sx = x * tile, sy = y * tile;
      const int ex = std::min(sx + tile, Wp), ey = std::min(sy + tile, Hp);
      const int sxp = std::max(sx - pad, 0), exp_ = std::min(ex + pad, Wp);
      const int syp = std::max(sy - pad, 0), eyp = std::min(ey + pad, Hp);
      TileBox b;
      memset(&b, 0, sizeof(b));
      b.src_y = syp; b.src_x = sxp;
      b.off_y = (sy - syp) * s; b.off_x = (sx - sxp) * s;
      b.dst_y = sy * s; b.dst_x = sx * s;
      b.paste_h = (ey - sy) * s; b.paste_w = (ex - sx) * s;
      classes[std::make_pair(eyp - syp, exp_ - sxp)].push_back(b);
    }
  // Crops of different shapes share an image as a CROP ATLAS: the crops of a group sit side by side (top-aligned, zero gap
  // columns between them) in atlas images of the group's canvas, everything outside the crops is zero on the way in and is
  // forced back to zero by every conv's epilogue (StreamParams::mask_hw), so each crop sees exactly the zero padding at its
  // own border that a run of its own would give it -- bit-identical, but the frame's tiles are one or two large launches
  // per conv instead of one small launch per shape class (1080p, tile 512: nine classes), and a row of the atlas fills
  // the kernel's 128-pixel strips instead of leaving every crop's last strip partly empty.  Groups collect crops of similar
  // height (tallest first; a crop joins while it is at least 90 % of the group's height); a group is cut into images of at
  // most kMaskRects crops.
  std::vector<std::pair<std::pair<int, int>, TileBox>> all;
  for (auto& kv : classes)
    for (const TileBox& b : kv.second) all.push_back(std::make_pair(kv.first, b));
  const int tdiv = (cfg->arch == SS4K_ARCH_RRDB && s == 2) ? 2 : 1;   // coarsest conv resolution = input / tdiv
  bool aligned = true;
  for (auto& e : all) aligned = aligned && e.first.first % tdiv == 0 && e.first.second % tdiv == 0;
  const bool merge = getenv("SS4K_TILE_EXACT_CLASSES") == nullptr && aligned;
  std::stable_sort(all.begin(), all.end(), [](const std::pair<std::pair<int, int>, TileBox>& a, const std::pair<std::pair<int, int>, TileBox>& b) {
    return a.first.first != b.first.first ? a.first.first > b.first.first : a.first.second > b.first.second; });
  for (auto& e : all) {
    TileBox b = e.second;
    b.crop_h = e.first.first; b.crop_w = e.first.second; b.img = 0; b.atlas_x = 0;
    bool placed = false;
    if (!groups.empty()) {
      TileGroup& g = groups.back();
      const bool same = b.crop_h == g.boxes[0].crop_h && b.crop_w == g.boxes[0].crop_w && g.boxes.back().crop_w == b.crop_w && g.boxes.back().crop_h == b.crop_h;
      if (merge ? b.crop_h * 10 >= g.hc * 9 : same) { g.boxes.push_back(b); placed = true; }
    }
    if (!placed) {
      groups.emplace_back();
      groups.back().hc = b.crop_h;
      groups.back().boxes.push_back(b);
    }
  }
  for (TileGroup& g : groups) {
    const int cnt = static_cast<int>(g.boxes.size());
    if (!merge) {   // one image per crop, no atlas (the classes are uniform)
      g.nimg = cnt; g.wc = g.boxes[0].crop_w;
      for (int k = 0; k < cnt; ++k) { g.boxes[k].img = k; g.boxes[k].atlas_x = 0; }
      continue;
    }
    g.nimg = (cnt + kMaskRects - 1) / kMaskRects;
    const int per = (cnt + g.nimg - 1) / g.nimg;
    const int gap = tdiv;   // one zero column at the coarsest resolution
    g.wc = 0;
    for (int k = 0; k < cnt; ++k) {
      const int im = k / per;
      const bool first = k % per == 0;
      g.boxes[k].img = im;
      g.boxes[k].atlas_x = first ? 0 : g.boxes[k - 1].atlas_x + g.boxes[k - 1].crop_w + gap;
      g.wc = std::max(g.wc, g.boxes[k].atlas_x + g.boxes[k].crop_w);
    }
  }
  return "";
}

static int create_tiled_plan(ss4k_ctx* ctx, const ss4k_plan_cfg* cfg, ss4k_plan** out_plan) {
  std::vector<TileGroup> groups;
  {
    std::string e = nv12_out_check(lite(cfg));
    if (e.empty()) e = layout_tiles(cfg, &groups);
    if (!e.empty()) return fail(ctx, SS4K_E_INVALID, e);
  }
  const int s = cfg->scale;
  // NV12 output: the tile classes paste uint8 RGB into a frame of the plan, converted once per run (crops need not have
  // NV12-compatible sizes)
  const bool nv12 = cfg->out_fmt == SS4K_FMT_NV12;
  std::unique_ptr<ss4k_plan> pl(new ss4k_plan());
  pl->ctx = ctx;
  pl->cfg = *cfg;
  pl->tiled = true;
  Program& P = pl->prog;
  P.in_fmt = cfg->in_fmt; P.out_fmt = cfg->out_fmt;
  P.in_n = cfg->n; P.in_c = 3; P.in_h = cfg->h; P.in_w = cfg->w;
  P.out_n = cfg->n; P.out_c = 3; P.out_h = cfg->h * s; P.out_w = cfg->w * s;
  for (auto& g : groups) {
    ss4k_plan::TileClass tc;
    tc.hc = g.hc; tc.wc = g.wc; tc.count = static_cast<int>(g.boxes.size()); tc.nimg = g.nimg;
    bool uniform = true;   // every image is exactly one crop of the canvas size: no mask needed
    for (const TileBox& b : g.boxes) uniform = uniform && b.crop_h == g.hc && b.crop_w == g.wc && b.atlas_x == 0;
    uniform = uniform && g.nimg == tc.count;
    ss4k_plan_cfg sub = *cfg;
    sub.tile = 0; sub.reserved[1] = 0;
    if (nv12) sub.out_fmt = SS4K_FMT_U8_NHWC;
    sub.reserved[5] = uniform ? 0 : 1;
    sub.n = cfg->n * tc.nimg; sub.h = tc.hc; sub.w = tc.wc;
    pl->tiles.push_back(tc);
    ss4k_plan::TileClass& t = pl->tiles.back();
    struct KV { std::vector<TileBox>& second; } kv{g.boxes};
    int rc = ss4k_plan_create(ctx, &sub, &t.sub);
    if (rc != SS4K_OK) {
      const std::string why = ctx->err;
      ss4k_plan_destroy(pl.release());
      return fail(ctx, rc, fmt("tile group %dx%d: %s", tc.hc, tc.wc, why.c_str()));
    }
    if (!uniform) {   // the crops of every atlas image of the batch (image index = img * N + n)
      std::vector<int32_t> hw(static_cast<size_t>(kMaskStride) * sub.n, 0);
      for (const TileBox& b : g.boxes)
        for (int n = 0; n < cfg->n; ++n) {
          int32_t* e = hw.data() + (static_cast<size_t>(b.img) * cfg->n + n) * kMaskStride;
          const int k = e[0]++;
          e[1 + 3 * k] = b.atlas_x; e[2 + 3 * k] = b.crop_w; e[3 + 3 * k] = b.crop_h;
        }
      if (cudaMemcpy(t.sub->d_mask, hw.data(), hw.size() * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess) {
        ss4k_plan_destroy(pl.release());
        return fail(ctx, SS4K_E_CUDA, "mask table upload");
      }
    }
    cudaError_t ce = cudaMalloc(&t.d_boxes, kv.second.size() * sizeof(TileBox));
    if (ce == cudaSuccess) ce = cudaMemcpy(t.d_boxes, kv.second.data(), kv.second.size() * sizeof(TileBox), cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMalloc(&t.d_in, t.sub->in_bytes + 256);
    if (ce == cudaSuccess) ce = cudaMalloc(&t.d_out, t.sub->out_bytes + 256);
    if (ce != cudaSuccess) {
      ss4k_plan_destroy(pl.release());
      return fail(ctx, SS4K_E_NOMEM, fmt("tiled plan buffers: %s", cudaGetErrorString(ce)));
    }
    P.flops += t.sub->prog.flops;
  }
  pl->in_bytes = fmt_bytes(P.in_fmt, P.in_n, P.in_c, P.in_h, P.in_w);
  pl->out_bytes = fmt_bytes(P.out_fmt, P.out_n, P.out_c, P.out_h, P.out_w);
  if (nv12 && cudaMalloc(&pl->nv12_rgb, fmt_bytes(SS4K_FMT_U8_NHWC, P.out_n, 3, P.out_h, P.out_w) + 256) != cudaSuccess) {
    ss4k_plan_destroy(pl.release());
    return fail(ctx, SS4K_E_NOMEM, "NV12 output: uint8 RGB frame");
  }
  cudaDeviceSynchronize();   // the tile boxes were uploaded on the NULL stream
  *out_plan = pl.release();
  return SS4K_OK;
}

// Host-only debug entry: the tile grid of a configuration and its crop atlases as JSON (tests/test_tiling_cpu.py).
int ss4k_debug_tile_layout(const ss4k_plan_cfg* cfg, char** out_json) {
  if (!cfg || !out_json) return fail(nullptr, SS4K_E_INVALID, "null argument");
  std::vector<TileGroup> groups;
  const std::string e = layout_tiles(cfg, &groups);
  if (!e.empty()) return fail(nullptr, SS4K_E_INVALID, e);
  std::string js = "{\"max_rects\":" + std::to_string(kMaskRects) + ",\"groups\":[";
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    const TileGroup& g = groups[gi];
    js += fmt("%s{\"hc\":%d,\"wc\":%d,\"nimg\":%d,\"boxes\":[", gi ? "," : "", g.hc, g.wc, g.nimg);
    for (size_t k = 0; k < g.boxes.size(); ++k) {
      const TileBox& b = g.boxes[k];
      js += fmt("%s{\"src_y\":%d,\"src_x\":%d,\"off_y\":%d,\"off_x\":%d,\"dst_y\":%d,\"dst_x\":%d,\"paste_h\":%d,\"paste_w\":%d,"
                "\"crop_h\":%d,\"crop_w\":%d,\"img\":%d,\"atlas_x\":%d}", k ? "," : "", b.src_y, b.src_x, b.off_y, b.off_x, b.dst_y, b.dst_x,
                b.paste_h, b.paste_w, b.crop_h, b.crop_w, b.img, b.atlas_x);
    }
    js += "]}";
  }
  js += "]}";
  *out_json = static_cast<char*>(malloc(js.size() + 1));
  memcpy(*out_json, js.c_str(), js.size() + 1);
  return SS4K_OK;
}

// Pitched NV12 surfaces (one allocation per frame, as a hardware decoder / encoder owns them) <-> the packed chunk
// [n, h*3/2, w] the plans read: two 2-D DMA copies per frame, stream-ordered.
static int nv12_surfaces(ss4k_ctx* ctx, const ss4k_nv12_surface* sf, int n, int h, int w, uint8_t* packed, bool pack, cudaStream_t st) {
  DeviceGuard dev_guard(ctx ? ctx->device : -1);
  if (!ctx || !sf || !packed || n <= 0 || h <= 0 || w <= 0 || (h % 2) || (w % 2)) return fail(ctx, SS4K_E_INVALID, "bad argument to ss4k_nv12_pack / ss4k_nv12_unpack");
  const size_t frame = static_cast<size_t>(h) * w * 3 / 2;
  for (int i = 0; i < n; ++i) {
    if (!sf[i].y || !sf[i].uv || sf[i].pitch_y < w || sf[i].pitch_uv < w) return fail(ctx, SS4K_E_INVALID, fmt("NV12 surface %d: null plane or pitch < width", i));
    uint8_t* py = packed + i * frame;
    uint8_t* puv = py + static_cast<size_t>(h) * w;
    if (pack) {
      CK(ctx, cudaMemcpy2DAsync(py, w, sf[i].y, sf[i].pitch_y, w, h, cudaMemcpyDeviceToDevice, st));
      CK(ctx, cudaMemcpy2DAsync(puv, w, sf[i].uv, sf[i].pitch_uv, w, h / 2, cudaMemcpyDeviceToDevice, st));
    } else {
      CK(ctx, cudaMemcpy2DAsync(sf[i].y, sf[i].pitch_y, py, w, w, h, cudaMemcpyDeviceToDevice, st));
      CK(ctx, cudaMemcpy2DAsync(sf[i].uv, sf[i].pitch_uv, puv, w, w, h / 2, cudaMemcpyDeviceToDevice, st));
    }
  }
  return SS4K_OK;
}
int ss4k_nv12_pack(ss4k_ctx* ctx, const ss4k_nv12_surface* surfaces, int n, int h, int w, void* packed_dev, void* cuda_stream) {
  return nv12_surfaces(ctx, surfaces, n, h, w, reinterpret_cast<uint8_t*>(packed_dev), true, reinterpret_cast<cudaStream_t>(cuda_stream));
}
int ss4k_nv12_unpack(ss4k_ctx* ctx, const void* packed_dev, const ss4k_nv12_surface* surfaces, int n, int h, int w, void* cuda_stream) {
  return nv12_surfaces(ctx, surfaces, n, h, w, const_cast<uint8_t*>(reinterpret_cast<const uint8_t*>(packed_dev)), false,
                       reinterpret_cast<cudaStream_t>(cuda_stream));
}

int ss4k_rgb_to_nv12(ss4k_ctx* ctx, const void* rgb_dev, void* nv12_dev, int n, int h, int w, void* cuda_stream) {
  DeviceGuard dev_guard(ctx ? ctx->device : -1);
  if (!ctx || !rgb_dev || !nv12_dev || n <= 0 || h <= 0 || w <= 0) return fail(ctx, SS4K_E_INVALID, "bad argument to ss4k_rgb_to_nv12");
  if (h % 2 || w % 4) return fail(ctx, SS4K_E_INVALID, "ss4k_rgb_to_nv12 needs h % 2 == 0 and w % 4 == 0");
  CK(ctx, rgb_to_nv12_launch(rgb_dev, nv12_dev, n, h, w, static_cast<cudaStream_t>(cuda_stream)));
  ctx->launches += 1;
  return SS4K_OK;
}

int ss4k_plan_out_shape(const ss4k_plan* pl, int32_t out_nchw[4]) {
  if (!pl || !out_nchw) return SS4K_E_INVALID;
  out_nchw[0] = pl->prog.out_n; out_nchw[1] = pl->prog.out_c; out_nchw[2] = pl->prog.out_h; out_nchw[3] = pl->prog.out_w;
  return SS4K_OK;
}
double ss4k_plan_flops(const ss4k_plan* pl) { return pl ? pl->prog.flops : 0.0; }
static int live_steps(const ss4k_plan* pl, int first, int last) {
  int n = 0;
  for (int si = first; si <= last; ++si)
    if (si != pl->fused_prep) ++n;
  return n;
}
// kernels one run launches (a layout step done by the first conv's loader launches nothing)
int ss4k_plan_launches(const ss4k_plan* pl) {
  if (!pl) return 0;
  int n = live_steps(pl, 0, static_cast<int>(pl->prog.steps.size()) - 1);
  for (const auto& t : pl->tiles) n += ss4k_plan_launches(t.sub) + 2;   // + gather and paste of the tile class
  if (pl->tiled && pl->nv12_rgb != nullptr) n += 1;                      // + the NV12 conversion of the pasted frame
  return n;
}
int ss4k_plan_graph_steps(const ss4k_plan* pl) {
  if (!pl) return 0;
  int n = pl->graph ? live_steps(pl, pl->graph_first, pl->graph_last) : 0;
  for (const auto& t : pl->tiles) n += ss4k_plan_graph_steps(t.sub);
  return n;
}
int ss4k_plan_steps(const ss4k_plan* pl) { return pl ? static_cast<int>(pl->prog.steps.size()) : 0; }
int ss4k_plan_io_bytes(const ss4k_plan* pl, int64_t* in_bytes, int64_t* out_bytes) {
  if (!pl) return SS4K_E_INVALID;
  if (in_bytes) *in_bytes = pl->in_bytes;
  if (out_bytes) *out_bytes = pl->out_bytes;
  return SS4K_OK;
}

int ss4k_run(ss4k_plan* pl, const void* in_dev, void* out_dev, void* cuda_stream) {
  if (!pl || !in_dev || !out_dev) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_run");
  ss4k_ctx* ctx = pl->ctx;
  DeviceGuard dev_guard(ctx->device);   // launches go to the engine's GPU whatever the calling thread's current device is
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  if (pl->tiled) {
    const Program& P = pl->prog;
    const bool nv12 = pl->nv12_rgb != nullptr;   // paste uint8 RGB into the plan's frame, convert it at the end
    for (auto& t : pl->tiles) {
      CK(ctx, tile_gather_launch(P.in_fmt, in_dev, t.d_in, t.d_boxes, t.count, t.nimg, P.in_n, 3, P.in_h, P.in_w, pl->cfg.reserved[1], t.hc, t.wc, st));
      int rc = ss4k_run(t.sub, t.d_in, t.d_out, cuda_stream);
      if (rc != SS4K_OK) return rc;
      CK(ctx, tile_paste_launch(nv12 ? SS4K_FMT_U8_NHWC : P.out_fmt, t.d_out, nv12 ? pl->nv12_rgb : out_dev, t.d_boxes, t.count, P.in_n, 3,
                                t.sub->prog.out_h, t.sub->prog.out_w, pl->cfg.scale, P.out_h, P.out_w, st));
      ctx->launches += 2;
    }
    if (nv12) {
      CK(ctx, rgb_to_nv12_launch(pl->nv12_rgb, out_dev, P.out_n, P.out_h, P.out_w, st));
      ctx->launches += 1;
    }
    return SS4K_OK;
  }
  const int ns = static_cast<int>(pl->prog.steps.size());
  for (int si = 0; si < ns; ++si) {
    if (pl->graph && si == pl->graph_first) {
      CK(ctx, cudaGraphLaunch(pl->graph, st));
      ctx->launches += live_steps(pl, pl->graph_first, pl->graph_last);
      si = pl->graph_last;
      continue;
    }
    int rc = run_step(pl, si, in_dev, out_dev, st);
    if (rc != SS4K_OK) return rc;
  }
  return SS4K_OK;
}

// The plan's first-layer activation tensor: where its layout step would write.  A producer that already has the frame
// on the device in float form (the service glue between denoiser and upscaler) writes it here itself and calls
// ss4k_run_act, which runs the plan without the layout step.
int ss4k_plan_input_act(ss4k_plan* pl, void** act_dev, int32_t* pitch, int32_t* unshuffle, int32_t* is_bf16) {
  if (!pl || !act_dev) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_plan_input_act");
  const Program& P = pl->prog;
  if (pl->tiled || P.steps.empty() || P.steps[0].kind != 0 || P.steps[0].prep.out_lo_buf >= 0 || pl->fused_prep >= 0)
    return fail(pl->ctx, SS4K_E_INVALID, "ss4k_plan_input_act: the plan has no plain layout step in front (tiled / split precision / frame-decoding plans)");
  const PrepSpec& p = P.steps[0].prep;
  *act_dev = pl->bufs[p.out_buf];
  if (pitch) *pitch = P.bufs[p.out_buf].pitch;
  if (unshuffle) *unshuffle = p.unshuffle;
  if (is_bf16) *is_bf16 = pl->cfg.act_mode == SS4K_ACT_BF16 ? 1 : 0;
  return SS4K_OK;
}

int ss4k_run_act(ss4k_plan* pl, void* out_dev, void* cuda_stream) {
  if (!pl || !out_dev) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_run_act");
  ss4k_ctx* ctx = pl->ctx;
  DeviceGuard dev_guard(ctx->device);
  void* act = nullptr;
  int rc = ss4k_plan_input_act(pl, &act, nullptr, nullptr, nullptr);
  if (rc != SS4K_OK) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const int ns = static_cast<int>(pl->prog.steps.size());
  for (int si = 1; si < ns; ++si) {
    if (pl->graph && si == pl->graph_first) {
      CK(ctx, cudaGraphLaunch(pl->graph, st));
      ctx->launches += live_steps(pl, pl->graph_first, pl->graph_last);
      si = pl->graph_last;
      continue;
    }
    rc = run_step(pl, si, nullptr, out_dev, st);
    if (rc != SS4K_OK) return rc;
  }
  return SS4K_OK;
}

int ss4k_run_host(ss4k_plan* pl, const void* in_host, void* out_host) {
  if (!pl || !in_host || !out_host) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_run_host");
  ss4k_ctx* ctx = pl->ctx;
  DeviceGuard dev_guard(ctx->device);
  if (!pl->stage_in) CK(ctx, cudaMalloc(&pl->stage_in, pl->in_bytes + 256));
  if (!pl->stage_out) CK(ctx, cudaMalloc(&pl->stage_out, pl->out_bytes + 256));
  CK(ctx, cudaMemcpyAsync(pl->stage_in, in_host, pl->in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  int rc = ss4k_run(pl, pl->stage_in, pl->stage_out, ctx->stream);
  if (rc != SS4K_OK) return rc;
  CK(ctx, cudaMemcpyAsync(out_host, pl->stage_out, pl->out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return check_kernel_health(ctx, cudaStreamSynchronize(ctx->stream), "ss4k_run_host");
}


// Pipelined host path: call i uses staging slot i & 1.  H2D on its own stream (after the kernels of call i-2 have
// consumed the slot), the plan on the engine stream, D2H on its own stream (after which the slot's output buffer may be
// overwritten by call i+2).
int ss4k_run_host_async(ss4k_plan* pl, const void* in_host, void* out_host) {
  if (!pl || !in_host || !out_host) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_run_host_async");
  ss4k_ctx* ctx = pl->ctx;
  DeviceGuard dev_guard(ctx->device);
  auto& pp = pl->pipe;
  if (!pp.init) {
    CK(ctx, cudaStreamCreateWithFlags(&pp.h2d, cudaStreamNonBlocking));
    CK(ctx, cudaStreamCreateWithFlags(&pp.d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CK(ctx, cudaMalloc(&pp.in[i], pl->in_bytes + 256));
      CK(ctx, cudaMalloc(&pp.out[i], pl->out_bytes + 256));
      CK(ctx, cudaEventCreateWithFlags(&pp.in_ready[i], cudaEventDisableTiming));
      CK(ctx, cudaEventCreateWithFlags(&pp.out_ready[i], cudaEventDisableTiming));
      CK(ctx, cudaEventCreateWithFlags(&pp.out_copied[i], cudaEventDisableTiming));
    }
    pp.init = true;
  }
  const int s = static_cast<int>(pp.calls & 1);
  const bool reused = pp.calls >= 2;
  ++pp.calls;
  if (reused) CK(ctx, cudaStreamWaitEvent(pp.h2d, pp.out_ready[s], 0));  // call i-2's kernels have read in[s]
  CK(ctx, cudaMemcpyAsync(pp.in[s], in_host, pl->in_bytes, cudaMemcpyHostToDevice, pp.h2d));
  CK(ctx, cudaEventRecord(pp.in_ready[s], pp.h2d));
  CK(ctx, cudaStreamWaitEvent(ctx->stream, pp.in_ready[s], 0));
  if (reused) CK(ctx, cudaStreamWaitEvent(ctx->stream, pp.out_copied[s], 0));  // call i-2's result has left out[s]
  int rc = ss4k_run(pl, pp.in[s], pp.out[s], ctx->stream);
  if (rc != SS4K_OK) return rc;
  CK(ctx, cudaEventRecord(pp.out_ready[s], ctx->stream));
  CK(ctx, cudaStreamWaitEvent(pp.d2h, pp.out_ready[s], 0));
  CK(ctx, cudaMemcpyAsync(out_host, pp.out[s], pl->out_bytes, cudaMemcpyDeviceToHost, pp.d2h));
  CK(ctx, cudaEventRecord(pp.out_copied[s], pp.d2h));
  return SS4K_OK;
}

int ss4k_plan_host_sync(ss4k_plan* pl) {
  if (!pl) return fail(nullptr, SS4K_E_INVALID, "null plan");
  ss4k_ctx* ctx = pl->ctx;
  if (pl->pipe.init) {
    CK(ctx, cudaStreamSynchronize(pl->pipe.h2d));
    int rc = check_kernel_health(ctx, cudaStreamSynchronize(ctx->stream), "ss4k_plan_host_sync");
    if (rc != SS4K_OK) return rc;
    CK(ctx, cudaStreamSynchronize(pl->pipe.d2h));
  }
  return SS4K_OK;
}

// Per-step timing of one plan run (no CUDA graph): a CUDA event between every step on `cuda_stream`.
// kind[i]: 0 prep / layout kernel, 1 row-streaming conv kernel, 2 tile conv kernel, 4 a layout step done by the first
// conv's loader.  Returns the number of steps.
int ss4k_plan_profile(ss4k_plan* pl, const void* in_dev, void* out_dev, void* cuda_stream, float* ms, double* flops,
                      int32_t* kind, int cap) {
  if (!pl || !in_dev || !out_dev || !ms || !flops || !kind) return fail(pl ? pl->ctx : nullptr, SS4K_E_INVALID, "null argument to ss4k_plan_profile");
  ss4k_ctx* ctx = pl->ctx;
  DeviceGuard dev_guard(ctx->device);
  if (pl->tiled) return fail(ctx, SS4K_E_INVALID, "ss4k_plan_profile: profile the tile classes' shapes as plans of their own");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const int ns = static_cast<int>(pl->prog.steps.size());
  if (cap < ns) return fail(ctx, SS4K_E_INVALID, "ss4k_plan_profile: arrays too small");
  std::vector<cudaEvent_t> ev(ns + 1);
  for (auto& e : ev) cudaEventCreate(&e);
  int rc = SS4K_OK;
  cudaEventRecord(ev[0], st);
  for (int si = 0; si < ns && rc == SS4K_OK; ++si) {
    rc = run_step(pl, si, in_dev, out_dev, st);
    cudaEventRecord(ev[si + 1], st);
  }
  if (rc == SS4K_OK) rc = check_kernel_health(ctx, cudaStreamSynchronize(st), "ss4k_plan_profile");
  for (int si = 0; si < ns && rc == SS4K_OK; ++si) {
    cudaEventElapsedTime(&ms[si], ev[si], ev[si + 1]);
    const Step& s = pl->prog.steps[si];
    flops[si] = s.kind == 1 ? s.conv.flops() : 0.0;
    if (s.kind == 2) { kind[si] = 0; continue; }   // the NV12 conversion of a two-step NV12 output: a colour kernel
    kind[si] = s.kind == 0 ? (si == pl->fused_prep ? 4 : 0) : (pl->convs[pl->step_conv[si]].stream ? 1 : 2);
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc == SS4K_OK ? ns : rc;
}

// ------------------------------------------------------------------------------------------------
// operator-level entry
int ss4k_conv3x3(ss4k_ctx* ctx, const ss4k_conv_desc* d, const float* x, const float* weight, const float* bias,
                 const float* slope, const float* residual, float* y, void* cuda_stream) {
  if (!ctx || !d || !x || !weight || !y) return fail(ctx, SS4K_E_INVALID, "null argument to ss4k_conv3x3");
  DeviceGuard dev_guard(ctx->device);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const bool bf16 = d->act_mode == SS4K_ACT_BF16;
  const bool split = d->act_mode == SS4K_ACT_F16_SPLIT;
  const int direct_f32 = d->reserved[0];
  const int in_pitch = round_up(d->cin, 16);
  const int npad = round_up(d->cout, 16);
  int oh = d->h, ow = d->w;
  if (d->mode == kModeUp2) { oh *= 2; ow *= 2; }
  if (d->mode == kModeS2) { oh /= 2; ow /= 2; }
  // weights to host
  HostTensor W, B, S;
  W.shape = {d->cout, d->cin, 3, 3};
  W.data.resize(static_cast<size_t>(d->cout) * d->cin * 9);
  CK(ctx, cudaMemcpyAsync(W.data.data(), weight, W.data.size() * 4, cudaMemcpyDeviceToHost, st));
  if (bias) { B.shape = {d->cout}; B.data.resize(d->cout); CK(ctx, cudaMemcpyAsync(B.data.data(), bias, d->cout * 4, cudaMemcpyDeviceToHost, st)); }
  if (slope) { S.shape = {d->cout}; S.data.resize(d->cout); CK(ctx, cudaMemcpyAsync(S.data.data(), slope, d->cout * 4, cudaMemcpyDeviceToHost, st)); }
  CK(ctx, cudaStreamSynchronize(st));
  // buffers: 0 in, 1 in_lo, 2 out, 3 res, 4 out_lo
  void* b[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  const size_t in_elems = static_cast<size_t>(d->n) * d->h * d->w * in_pitch;
  const int out_ch_pitch = d->pixel_shuffle == 2 ? npad / 4 : npad;
  const int ooh = d->pixel_shuffle == 2 ? oh * 2 : oh, oow = d->pixel_shuffle == 2 ? ow * 2 : ow;
  const size_t out_elems = static_cast<size_t>(d->n) * ooh * oow * out_ch_pitch;
  auto cleanup = [&]() { for (void* q : b) if (q) cudaFree(q); };
  CK(ctx, cudaMalloc(&b[0], in_elems * 2 + 256));
  if (split) CK(ctx, cudaMalloc(&b[1], in_elems * 2 + 256));
  CK(ctx, cudaMalloc(&b[2], out_elems * 2 + 256));
  if (split) CK(ctx, cudaMalloc(&b[4], out_elems * 2 + 256));
  CK(ctx, prep_launch(SS4K_FMT_F32_NCHW, x, b[0], b[1], d->n, d->cin, d->h, d->w, in_pitch, 1, -1, 0.f, bf16, st));
  ctx->launches++;
  const bool ps_f32 = d->pixel_shuffle > 0 && d->pixel_shuffle != 2;
  const int res_c = d->pixel_shuffle == 2 ? d->cout / 4 : d->cout;
  if (residual) {
    CK(ctx, cudaMalloc(&b[3], out_elems * 2 + 256));
    CK(ctx, prep_launch(SS4K_FMT_F32_NCHW, residual, b[3], nullptr, d->n, res_c, ooh, oow, out_ch_pitch, 1, -1, 0.f, bf16, st));
    ctx->launches++;
  }
  ConvSpec cs;
  cs.name = "op"; cs.wname = "w"; cs.mode = d->mode; cs.n = d->n; cs.cin = d->cin; cs.cout = d->cout;
  cs.in_buf = 0; cs.in_lo_buf = split ? 1 : kBufNone; cs.in_h = d->h; cs.in_w = d->w; cs.in_pitch = in_pitch;
  cs.act = d->act; cs.alpha = d->alpha; cs.split = split ? 1 : 0;
  if (residual) { cs.res1_buf = 3; cs.res1_pitch = out_ch_pitch; cs.beta1 = d->beta; }
  if (ps_f32) {
    cs.out_mode = kOutPSNCHWF32; cs.out_buf = kBufExternalOut; cs.ps_r = d->pixel_shuffle; cs.out_h = oh; cs.out_w = ow;
  } else if (d->pixel_shuffle == 2) {
    cs.out_mode = kOutPS2NHWC; cs.out_buf = 2; cs.out_pitch = out_ch_pitch; cs.out_h = ooh; cs.out_w = oow; cs.wperm = 1;
    cs.out_lo_buf = split ? 4 : kBufNone;
  } else if (direct_f32) {
    cs.out_mode = kOutNCHWF32; cs.out_buf = kBufExternalOut; cs.out_h = oh; cs.out_w = ow;
  } else {
    cs.out_mode = kOutNHWC; cs.out_buf = 2; cs.out_pitch = npad; cs.out_h = oh; cs.out_w = ow;
    cs.out_lo_buf = split ? 4 : kBufNone;
  }
  ConvExec ex;
  auto bufptr = [&](int id) -> void* { return id >= 0 ? b[id] : nullptr; };
  int rc = materialize_conv(ctx, cs, W, bias ? &B : nullptr, slope ? &S : nullptr, d->act_mode, bufptr, &ex);
  if (rc != SS4K_OK) { free_conv(ex); cleanup(); return rc; }
  cudaError_t ce = cudaDeviceSynchronize();   // packed weights were uploaded on the NULL stream
  if (ce == cudaSuccess) ce = launch_exec(ex, y, st);
  ctx->launches++;
  if (ce == cudaSuccess && !ex.ext_out) {
    ce = unprep_launch(b[2], b[4], y, d->n, res_c, ooh, oow, out_ch_pitch, 0, bf16, st);
    ctx->launches++;
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
  rc = check_kernel_health(ctx, ce, "ss4k_conv3x3");
  free_conv(ex);
  cleanup();
  return rc;
}

// ------------------------------------------------------------------------------------------------
// Host-only debug entry: run the weight packer and return its schedule as JSON + the packed weights
// as floats.  tests/test_pack_cpu.py emulates the kernel's MMA schedule from this on the CPU.
int ss4k_debug_pack(const ss4k_conv_desc* d, int in_pitch, int in_coff, int wperm, const float* w_host,
                    const float* bias_host, const float* slope_host, char** out_json, float** out_packed,
                    int64_t* out_count) {
  if (!d || !w_host || !out_json || !out_packed || !out_count) return fail(nullptr, SS4K_E_INVALID, "null argument");
  ConvSpec cs;
  cs.name = "dbg"; cs.wname = "w"; cs.mode = d->mode; cs.n = d->n; cs.cin = d->cin; cs.cout = d->cout;
  cs.in_h = d->h; cs.in_w = d->w; cs.in_pitch = in_pitch; cs.in_coff = in_coff; cs.wperm = wperm;
  cs.split = d->act_mode == SS4K_ACT_F16_SPLIT ? 1 : 0;
  HostTensor W, B, S;
  W.shape = {d->cout, d->cin, 3, 3};
  W.data.assign(w_host, w_host + static_cast<size_t>(d->cout) * d->cin * 9);
  if (bias_host) { B.shape = {d->cout}; B.data.assign(bias_host, bias_host + d->cout); }
  if (slope_host) { S.shape = {d->cout}; S.data.assign(slope_host, slope_host + d->cout); }
  const bool bf16 = d->act_mode == SS4K_ACT_BF16;
  if (d->reserved[6] == 1) {  // row-streaming kernel layout
    StreamPacked sp;
    cs.act = d->act; cs.alpha = d->alpha != 0.f ? d->alpha : 1.f;
    if (!stream_config(cs, &sp)) return fail(nullptr, SS4K_E_INVALID, "conv is not eligible for the row-streaming kernel");
    std::string es = pack_weights_stream(cs, W, bias_host ? &B : nullptr, slope_host ? &S : nullptr, bf16, &sp);
    if (!es.empty()) return fail(nullptr, SS4K_E_WEIGHTS, es);
    std::string js = fmt("{\"kernel\":\"stream\",\"nout\":%d,\"chunks\":%d,\"nkb\":%d,\"npad\":%d,\"a_slots\":%d,\"acc_slots\":%d,\"w_rows\":%d,\"nks\":[",
                         sp.nout, sp.chunks, sp.nkb, sp.npad_total, sp.a_slots, sp.acc_slots, sp.bias_row0);
    for (int i = 0; i < sp.nkb; ++i) js += fmt("%s%d", i ? "," : "", sp.nks[i]);
    js += fmt("],\"stride2\":%d,\"nkx\":%d,\"ksm\":[", sp.stride2, sp.nkx);
    for (int i = 0; i < sp.nkb; ++i) js += fmt("%s[%d,%d]", i ? "," : "", sp.ksm[i][0], sp.ksm[i][1]);
    js += fmt("],\"nwt\":%d,\"wt\":[", sp.nwt);
    for (int i = 0; i < sp.nkb; ++i) js += fmt("%s%d", i ? "," : "", sp.wt[i]);
    js += "],\"src_kb\":[";
    for (int i = 0; i < sp.nkb; ++i) js += fmt("%s%d", i ? "," : "", sp.src_kb[i]);
    js += "],\"bias\":[";
    for (size_t i = 0; i < sp.bias.size(); ++i) js += fmt("%s%.9g", i ? "," : "", sp.bias[i]);
    js += "],\"bias_f\":[";
    for (size_t i = 0; i < sp.bias_f.size(); ++i) js += fmt("%s%.9g", i ? "," : "", sp.bias_f[i]);
    js += "],\"slope\":[";
    for (size_t i = 0; i < sp.slope.size(); ++i) js += fmt("%s%.9g", i ? "," : "", sp.slope[i]);
    js += "]}";
    *out_json = static_cast<char*>(malloc(js.size() + 1));
    memcpy(*out_json, js.c_str(), js.size() + 1);
    *out_count = static_cast<int64_t>(sp.w.size());
    *out_packed = static_cast<float*>(malloc(sp.w.size() * sizeof(float)));
    for (size_t i = 0; i < sp.w.size(); ++i) (*out_packed)[i] = h2f(sp.w[i], bf16);
    return SS4K_OK;
  }
  PackedWeights pw;
  std::string e = pack_weights(cs, W, bias_host ? &B : nullptr, slope_host ? &S : nullptr, bf16, &pw);
  if (!e.empty()) return fail(nullptr, SS4K_E_WEIGHTS, e);
  int AH = d->h, AW = d->w;
  if (d->mode == kModeS2) { AH /= 2; AW /= 2; }
  TileCfg t;
  const int dm = d->reserved[1];
  e = configure_tiles(dm, 148, d->n, AH, AW, pw.npad_total, pw.ntaps, pw.nsub, pw.max_dr, pw.nkb, &t);
  if (!e.empty()) return fail(nullptr, SS4K_E_INVALID, e);
  std::string js = "{";
  js += fmt("\"nkb\":%d,\"ntaps\":%d,\"nsub\":%d,\"max_dr\":%d,\"npad\":%d,", pw.nkb, pw.ntaps, pw.nsub, pw.max_dr, pw.npad_total);
  js += fmt("\"R\":%d,\"n_cta\":%d,\"n_chunks\":%d,\"acc_stride\":%d,\"tiles_x\":%d,\"tiles_y\":%d,\"n_tiles\":%d,", t.R, t.n_cta, t.n_chunks, t.acc_stride, t.tiles_x, t.tiles_y, t.n_tiles);
  js += fmt("\"a_slots\":%d,\"a_slot_bytes\":%d,\"w_slots\":%d,\"w_slot_bytes\":%d,\"w_resident\":%d,", t.a_slots, t.a_slot_bytes, t.w_slots, t.w_slot_bytes, t.w_resident);
  js += "\"kb\":[";
  for (int i = 0; i < pw.nkb; ++i) js += fmt("%s[%d,%d,%d]", i ? "," : "", pw.kb[i].tmap, pw.kb[i].c0, pw.kb[i].p);
  js += "],\"taps\":[";
  for (int i = 0; i < pw.ntaps; ++i) js += fmt("%s[%d,%d,%d]", i ? "," : "", pw.taps[i].dr, pw.taps[i].shift, pw.taps[i].sub);
  js += "],\"mask\":[";
  for (int i = 0; i < pw.nkb; ++i) {
    js += i ? ",[" : "[";
    for (int j = 0; j < pw.ntaps; ++j) js += fmt("%s%d", j ? "," : "", pw.mask[static_cast<size_t>(i) * kMaxTaps + j]);
    js += "]";
  }
  js += "],\"bias\":[";
  for (size_t i = 0; i < pw.bias.size(); ++i) js += fmt("%s%.9g", i ? "," : "", pw.bias[i]);
  js += "],\"slope\":[";
  for (size_t i = 0; i < pw.slope.size(); ++i) js += fmt("%s%.9g", i ? "," : "", pw.slope[i]);
  js += "]}";
  *out_json = static_cast<char*>(malloc(js.size() + 1));
  memcpy(*out_json, js.c_str(), js.size() + 1);
  *out_count = static_cast<int64_t>(pw.w.size());
  *out_packed = static_cast<float*>(malloc(pw.w.size() * sizeof(float)));
  for (size_t i = 0; i < pw.w.size(); ++i) (*out_packed)[i] = h2f(pw.w[i], bf16);
  return SS4K_OK;
}

// ------------------------------------------------------------------------------------------------
// Debug / profiling entry: time `iters` launches of one conv (buffers hold zeros) with CUDA events.
// dbg_flags: see ConvParams::dbg_flags.  slab_pitch: channel pitch of the input tensor (>= cin).
int ss4k_debug_bench_conv(ss4k_ctx* ctx, const ss4k_conv_desc* d, int slab_pitch, int dbg_flags, int iters,
                          float* ms_per_launch, char** out_json) {
  if (!ctx || !d || !ms_per_launch) return fail(ctx, SS4K_E_INVALID, "null argument");
  DeviceGuard dev_guard(ctx->device);
  const bool bf16 = d->act_mode == SS4K_ACT_BF16;
  const int in_pitch = slab_pitch > 0 ? slab_pitch : round_up(d->cin, 16);
  const int npad = round_up(d->cout, 16);
  int oh = d->h, ow = d->w;
  if (d->mode == kModeUp2) { oh *= 2; ow *= 2; }
  if (d->mode == kModeS2) { oh /= 2; ow /= 2; }
  HostTensor W;
  W.shape = {d->cout, d->cin, 3, 3};
  W.data.assign(static_cast<size_t>(d->cout) * d->cin * 9, 0.01f);
  if (d->reserved[6] == 1) {  // random weights (power measurements: MMA energy depends on the operand values)
    uint32_t s = 2463534242u;
    for (auto& v : W.data) { s = s * 1664525u + 1013904223u; v = (((s >> 8) & 0xFFFF) / 65536.0f - 0.5f) * 0.1f; }
  }
  void* b[3] = {nullptr, nullptr, nullptr};
  const size_t in_bytes = static_cast<size_t>(d->n) * d->h * d->w * in_pitch * 2 + 256;
  const size_t out_bytes = static_cast<size_t>(d->n) * oh * ow * npad * 2 + 256;
  CK(ctx, cudaMalloc(&b[0], in_bytes));
  CK(ctx, cudaMalloc(&b[1], out_bytes));
  CK(ctx, cudaMalloc(&b[2], out_bytes));
  CK(ctx, cudaMemset(b[0], 0, in_bytes));
  CK(ctx, cudaMemset(b[2], 0, out_bytes));
  if (d->reserved[6] == 1) {  // random activations in (-1, 1)
    std::vector<uint16_t> hx(in_bytes / 2);
    uint32_t s = 88172645u;
    for (auto& v : hx) { s = s * 1664525u + 1013904223u; v = f2h((((s >> 8) & 0xFFFF) / 32768.0f - 1.0f), bf16); }
    CK(ctx, cudaMemcpy(b[0], hx.data(), hx.size() * 2, cudaMemcpyHostToDevice));
  }
  ConvSpec cs;
  cs.name = "bench"; cs.wname = "w"; cs.mode = d->mode; cs.n = d->n; cs.cin = d->cin; cs.cout = d->cout;
  cs.in_buf = 0; cs.in_h = d->h; cs.in_w = d->w; cs.in_pitch = in_pitch;
  cs.act = d->act; cs.alpha = d->alpha;
  cs.out_mode = kOutNHWC; cs.out_buf = 1; cs.out_pitch = npad; cs.out_h = oh; cs.out_w = ow;
  if (d->beta != 0.f) { cs.res1_buf = 2; cs.res1_pitch = npad; cs.beta1 = d->beta; }
  ConvExec ex;
  auto bufptr = [&](int id) -> void* { return id >= 0 ? b[id] : nullptr; };
  int rc = materialize_conv(ctx, cs, W, nullptr, nullptr, d->act_mode, bufptr, &ex);
  if (rc == SS4K_OK) {
    long long* d_trace = nullptr;
    if (ex.stream && d->reserved[7] == 1) {
      cudaMalloc(&d_trace, sizeof(long long) * 128 * 148);
      cudaMemset(d_trace, 0, sizeof(long long) * 128 * 148);
    }
    void* d_src = nullptr;
    if (ex.stream && d->reserved[1] != 0 && in_pitch == 16 && d->mode == kModeConv3) {  // frame-format source decoded by the kernel
      const size_t sb = static_cast<size_t>(d->n) * d->h * d->w * 3;
      cudaMalloc(&d_src, sb);
      cudaMemset(d_src, 128, sb);
      ex.sp.src = reinterpret_cast<const uint8_t*>(d_src);
      ex.sp.src_fmt = d->reserved[1]; ex.sp.src_fill_ch = 3; ex.sp.src_fill = 0.075f;
      ex.sp.src_out = reinterpret_cast<uint16_t*>(b[0]);
      ex.sp.src_out_lo = nullptr;
    }
    if (ex.stream) {
      ex.sp.dbg_flags = dbg_flags;
      if (d->reserved[3] > 0) ex.sp.a_slots = std::min(ex.sp.a_slots, d->reserved[3]);
      if (d->reserved[4] > 0) ex.sp.acc_slots = std::max(4, std::min(ex.sp.acc_slots, d->reserved[4]));
      if (d->reserved[5] > 0) ex.grid = std::min(ex.grid, d->reserved[5]);
    } else {
      ex.p.dbg_flags = dbg_flags;
      if (d->reserved[2] > 0) {  // override rows per tile
        ex.p.R = d->reserved[2];
        ex.p.tiles_y = (ex.p.H + ex.p.R - 1) / ex.p.R;
        ex.p.n_tiles = ex.p.n_img * ex.p.tiles_y * ex.p.tiles_x * ex.p.n_chunks;
        ex.grid = std::min(ex.p.n_tiles, ctx->nsm);
      }
      if (d->reserved[3] > 0) ex.p.a_slots = std::min(ex.p.a_slots, d->reserved[3]);
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaError_t ce = cudaSuccess;
    for (int i = 0; i < 3 && ce == cudaSuccess; ++i) ce = launch_exec(ex, nullptr, ctx->stream);
    cudaEventRecord(e0, ctx->stream);
    for (int i = 0; i < iters && ce == cudaSuccess; ++i) ce = launch_exec(ex, nullptr, ctx->stream);
    cudaEventRecord(e1, ctx->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    rc = check_kernel_health(ctx, ce, "ss4k_debug_bench_conv");
    float ms = 0.f;
    if (rc == SS4K_OK) cudaEventElapsedTime(&ms, e0, e1);
    *ms_per_launch = ms / std::max(1, iters);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    ctx->launches += iters + 3;
    std::string trace_js;
    if (d_trace != nullptr) {  // one extra traced launch: clock64 stamps of CTA 0 and the last CTA, relative to entry
      cudaMemset(d_trace, 0, sizeof(long long) * 128 * 148);
      ex.sp.trace = d_trace;
      launch_exec(ex, nullptr, ctx->stream);
      cudaStreamSynchronize(ctx->stream);
      ex.sp.trace = nullptr;
      std::vector<long long> h(128 * 148);
      cudaMemcpy(h.data(), d_trace, sizeof(long long) * 128 * 148, cudaMemcpyDeviceToHost);
      cudaFree(d_trace);
      trace_js = ",\"trace\":[";
      for (int b : {0, ex.grid / 2, ex.grid - 1}) {
        trace_js += (b == 0 ? "[" : ",[");
        for (int i = 0; i < 128; ++i) trace_js += fmt("%s%lld", i ? "," : "", h[b * 128 + i] ? h[b * 128 + i] - h[b * 128] : -1LL);
        trace_js += "]";
      }
      trace_js += "]";
    }
    if (out_json) {
      std::string js;
      if (ex.stream)
        js = fmt("{\"kernel\":\"stream\",\"nout\":%d,\"chunks\":%d,\"grid\":%d,\"a_slots\":%d,\"acc_slots\":%d,\"nkb\":%d,\"units\":%d}",
                 ex.nout, ex.sp.chunks, ex.grid, ex.sp.a_slots, ex.sp.acc_slots, ex.sp.nkb, ex.sp.total_units);
      else
        js = fmt("{\"kernel\":\"tile\",\"R\":%d,\"n_tiles\":%d,\"grid\":%d,\"a_slots\":%d,\"w_slots\":%d,\"w_resident\":%d,\"nkb\":%d,\"n_cta\":%d,\"n_chunks\":%d}",
                 ex.p.R, ex.p.n_tiles, ex.grid, ex.p.a_slots, ex.p.w_slots, ex.p.w_resident, ex.p.nkb, ex.p.n_cta, ex.p.n_chunks);
      if (!trace_js.empty()) js.insert(js.size() - 1, trace_js);
      *out_json = static_cast<char*>(malloc(js.size() + 1));
      memcpy(*out_json, js.c_str(), js.size() + 1);
    }
    if (d_src) cudaFree(d_src);
  }
  free_conv(ex);
  for (void* q : b) if (q) cudaFree(q);
  return rc;
}

// Start-up self-probe: one small 64->64 conv through the tcgen05 path against the naive direct
// kernel.  Decides which shared-memory-descriptor addressing mode this GPU/driver honours.
static int self_probe(ss4k_ctx* ctx) {
  const int N = 1, H = 5, W = 200, C = 64;
  std::vector<float> hx(static_cast<size_t>(N) * C * H * W), hw(static_cast<size_t>(C) * C * 9), hb(C);
  uint32_t s = 12345u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return ((s >> 8) & 0xFFFF) / 65536.0f - 0.5f; };
  for (auto& v : hx) v = rnd();
  for (auto& v : hw) v = h2f(f2h(rnd() * 0.2f, false), false);
  for (auto& v : hb) v = rnd();
  float *dx = nullptr, *dw = nullptr, *db = nullptr, *dy = nullptr, *dr = nullptr;
  void* dx16 = nullptr;
  const size_t osz = static_cast<size_t>(N) * C * H * W;
  CK(ctx, cudaMalloc(&dx, hx.size() * 4));
  CK(ctx, cudaMalloc(&dw, hw.size() * 4));
  CK(ctx, cudaMalloc(&db, hb.size() * 4));
  CK(ctx, cudaMalloc(&dy, osz * 4));
  CK(ctx, cudaMalloc(&dr, osz * 4));
  CK(ctx, cudaMalloc(&dx16, static_cast<size_t>(N) * H * W * C * 2 + 256));
  CK(ctx, cudaMemcpy(dx, hx.data(), hx.size() * 4, cudaMemcpyHostToDevice));
  CK(ctx, cudaMemcpy(dw, hw.data(), hw.size() * 4, cudaMemcpyHostToDevice));
  CK(ctx, cudaMemcpy(db, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice));
  // cudaMemcpy from pageable memory returns once the data is staged: its DMA runs on the NULL stream, which the engine's
  // non-blocking stream does not wait for (seen as wrong probe results when other processes keep the copy engine busy)
  CK(ctx, cudaDeviceSynchronize());
  ss4k_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.struct_size = sizeof(d); d.n = N; d.h = H; d.w = W; d.cin = C; d.cout = C; d.alpha = 1.f;
  d.reserved[0] = 1;
  int rc = ss4k_conv3x3(ctx, &d, dx, dw, db, nullptr, nullptr, dy, ctx->stream);
  if (rc == SS4K_OK) {
    cudaError_t ce = prep_launch(SS4K_FMT_F32_NCHW, dx, dx16, nullptr, N, C, H, W, C, 1, -1, 0.f, 0, ctx->stream);
    if (ce == cudaSuccess) ce = ref_conv3x3_launch(dx16, dw, db, dr, N, H, W, C, C, C, 0, ctx->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    rc = check_kernel_health(ctx, ce, "self-probe reference");
  }
  if (rc == SS4K_OK) {
    std::vector<float> y(osz), r(osz);
    cudaMemcpy(y.data(), dy, osz * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(r.data(), dr, osz * 4, cudaMemcpyDeviceToHost);
    double maxref = 0, maxerr = 0;
    for (size_t i = 0; i < osz; ++i) {
      maxref = std::max(maxref, static_cast<double>(std::fabs(r[i])));
      const double e = std::fabs(static_cast<double>(y[i]) - r[i]);
      if (!(e <= maxerr)) maxerr = e;  // also catches NaN
    }
    if (!(maxerr <= 2e-3 * maxref + 1e-3))
      rc = fail(ctx, SS4K_E_SELFTEST, fmt("max|err| %.4g vs max|ref| %.4g", maxerr, maxref));
  }
  cudaFree(dx); cudaFree(dw); cudaFree(db); cudaFree(dy); cudaFree(dr); cudaFree(dx16);
  return rc;
}

}  // extern "C"

#include "bsvd_stream.inc"
