// Host-side layer programs: a network is lowered to a list of buffers and steps (prep + convs with
// fused epilogues).  This part is pure host code (no CUDA calls) so the planner can be checked on a
// CPU-only box: ss4k_plan_dry() dumps a program as JSON and tests/test_program_cpu.py interprets it
// with torch against the oracle.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

namespace ss4k {

constexpr int kBufExternalIn = -2;   // caller's input pointer
constexpr int kBufExternalOut = -3;  // caller's output pointer
constexpr int kBufNone = -1;

struct BufSpec {
  std::string name;
  int n = 0, h = 0, w = 0, pitch = 0;  // NHWC, 16-bit elements
  bool zero_init = false;
  size_t bytes() const { return static_cast<size_t>(n) * h * w * pitch * 2 + 256; }
};

struct PrepSpec {
  int in_fmt = 0;       // SS4K_FMT_*
  int c = 3;            // source channels
  int h = 0, w = 0;     // source frame size
  int n = 1;
  int n0 = 0;           // first frame of the clip this step processes (BSVD chunks with a temporal halo, bsvd_program.cpp)
  int unshuffle = 1;    // pixel_unshuffle factor
  int out_buf = kBufNone, out_lo_buf = kBufNone;
  int fill_ch = -1;     // channel receiving a constant (BSVD noise map), or -1
  float fill_val = 0.f;
};

struct ConvSpec {
  std::string name;
  std::string wname, bname, sname;  // state-dict keys: weight, bias, PReLU slope ("" = none)
  float const_slope = 0.f;          // LeakyReLU slope when act == 1 and sname is empty
  int mode = 0;                     // ConvMode
  int n = 1;
  int n0 = 0, n_total = 0;          // BSVD chunk with halo: this step runs frames [n0, n0 + n) of the n_total-frame tensors (0: n0 = 0, all)
  int cin = 0, cout = 0;
  int in_buf = kBufNone, in_lo_buf = kBufNone;
  int in_h = 0, in_w = 0, in_pitch = 0, in_coff = 0;
  int act = 0;                      // ActKind
  float alpha = 1.f, beta1 = 0.f, beta2 = 0.f;
  int res1_buf = kBufNone, res1_pitch = 0, res1_coff = 0;
  int res2_buf = kBufNone, res2_pitch = 0, res2_coff = 0;
  int res1_lo_buf = kBufNone, res2_lo_buf = kBufNone;  // split mode: low halves of the residual tensors
  int out_mode = 0;                 // OutMode
  int out_buf = kBufNone, out_lo_buf = kBufNone, out2_buf = kBufNone, out3_buf = kBufNone;
  int out_pitch = 0, out_coff = 0;
  int out_h = 0, out_w = 0;         // see Epilogue::out_h
  int ps_r = 0, fold = 0, round_u8 = 0;
  int base_buf = kBufNone, base_pitch = 0;
  int wperm = 0;                    // 1: permute output channels (c,a,b) -> (a,b,c) for PixelShuffle(2)
  int split = 0;                    // 1: fp16 hi/lo split operands (3 MMAs per product)
  int neg_first = 0;                // negate weights and bias of the first k output channels (BSVD none_minus)
  int res1_nch = 0;                 // > 0: add only the first k channels of res1
  int tshift = 0;                   // 1: temporal-shift scatter store with fold = `fold` (time == batch index)
  int in_ring = 0, out_ring = 0;    // BSVD streaming: images (ring slots) of the input / output tensors (0: n)
  int up2_store = 0;                // 1: store every output pixel 2x2 times: the destination is the nearest-x2 upsampled image
  int discard_buf = kBufNone;       // tensor whose lines (bit l of discard_mask: 128-byte line l of every pixel) are dead:
  int discard_mask = 0;             //   dropped from L2 without write-back by this conv (no later step reads them)
  int discard_pitch = 0;            //   channel pitch of that tensor (16-bit elements; a multiple of 64 = whole lines)
  long long discard_npx = 0;        //   its pixel count
  int old_cin = 0;                  // input channels [0, old_cin) were written at least two steps ago (StreamParams::early_kb_mask)
  int l2_in = 0, l2_out = 0;        // L2 eviction priority hints of the loads / stores (StreamParams::l2_in / l2_out)
  double flops() const;
};

struct Step {
  int kind = 0;  // 0 prep, 1 conv, 2 uint8 RGB -> NV12 of the plan's output (added by the engine: NV12 output whose
                 //   last conv does not store NV12 itself, engine.cu::ss4k_plan_create)
  PrepSpec prep;
  ConvSpec conv;
};

struct Program {
  std::vector<BufSpec> bufs;
  std::vector<Step> steps;
  int out_n = 0, out_c = 0, out_h = 0, out_w = 0;
  int in_n = 0, in_c = 0, in_h = 0, in_w = 0;
  int in_fmt = 0, out_fmt = 0;
  double flops = 0;
  int add_buf(const std::string& name, int n, int h, int w, int pitch, bool zero = false) {
    BufSpec b;
    b.name = name; b.n = n; b.h = h; b.w = w; b.pitch = pitch; b.zero_init = zero;
    bufs.push_back(b);
    return static_cast<int>(bufs.size()) - 1;
  }
  void add_conv(const ConvSpec& c) {
    Step s; s.kind = 1; s.conv = c; steps.push_back(s);
    flops += c.flops();
  }
  void add_prep(const PrepSpec& p) {
    Step s; s.kind = 0; s.prep = p; steps.push_back(s);
  }
  std::string to_json() const;
};

struct PlanCfgLite {
  int arch, n, h, w, scale, depth, tile, tile_pad, act_mode, in_fmt, out_fmt;
  int bsvd_stream = 0;
  int own_lo = 0, own_hi = 0;  // BSVD: frames of the clip whose result is wanted (0, 0: all); the others are temporal halo
  float bsvd_noise = 0.f;  // noise-map value for 3-channel frame inputs (uint8 NHWC / NV12)  // 1: BSVD program for the streaming engine (separate buffers for temp1 / temp2)
};

// returns "" on success, else an error message
std::string build_program(const PlanCfgLite& cfg, Program* out);
// out_fmt SS4K_FMT_NV12: RRDBNet only, output height even and width divisible by 4 ("" when fine or not NV12)
std::string nv12_out_check(const PlanCfgLite& cfg);

}  // namespace ss4k
