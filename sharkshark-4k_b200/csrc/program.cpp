// Network -> layer program lowering (host only, no CUDA).  See program.h.
//
// Reference semantics restated here (all paths relative to the reference tree):
//   SRVGGNetCompact.forward   src/upscale/model/realesrgan/factory.py:71-82
//   RRDBNet.forward           basicsr/archs/rrdbnet_arch.py (un-vendored pip dependency, call sites
//                             factory.py:113-125; restated in SURVEY.md Appendix A)
//   BSVD / DenBlock           src/upscale/model/bsvd/model.py:353-442,467-588
#include "program.h"

#include <sstream>

#include "conv_params.h"

namespace ss4k {

double ConvSpec::flops() const {
  // algorithmic FLOPs: 2*Cin*Cout*9*Hout*Wout with true channel counts (SURVEY.md section 8d)
  double ho = in_h, wo = in_w;
  if (mode == kModeUp2) { ho *= 2; wo *= 2; }
  if (mode == kModeS2) { ho /= 2; wo /= 2; }
  return 2.0 * cin * cout * 9.0 * ho * wo * n;
}

namespace {

int round_up(int a, int b) { return (a + b - 1) / b * b; }

int final_out_mode(int out_fmt) {
  switch (out_fmt) {
    case 0: return kOutNCHWF32;
    case 1: return kOutNCHWF16;
    case 2: return kOutU8NHWC;
    case 3: return kOutNV12;
    default: return -1;
  }
}

// ------------------------------------------------------------------ SRVGGNetCompact
std::string build_srvgg(const PlanCfgLite& c, Program* P) {
  const int s = c.scale;
  if (s != 2 && s != 4 && s != 1 && s != 3) return "SRVGG: unsupported upscale";
  if (c.out_fmt != 0 && c.out_fmt != 1) return "SRVGG: output is float / half NCHW (the colour-match glue reads it; no uint8 / NV12 output)";
  const int nf = 64, nconv = c.depth > 0 ? c.depth : 16;
  const int cl = 3 * s * s;
  P->in_n = c.n; P->in_c = 3; P->in_h = c.h; P->in_w = c.w;
  P->out_n = c.n; P->out_c = 3; P->out_h = c.h * s; P->out_w = c.w * s;
  const int in16 = P->add_buf("in16", c.n, c.h, c.w, 16);
  const int fa = P->add_buf("featA", c.n, c.h, c.w, nf);
  const int fb = P->add_buf("featB", c.n, c.h, c.w, nf);
  PrepSpec pp;
  pp.in_fmt = c.in_fmt; pp.c = 3; pp.h = c.h; pp.w = c.w; pp.n = c.n; pp.out_buf = in16;
  P->add_prep(pp);
  int cur = in16, cur_pitch = 16, cur_c = 3;
  for (int i = 0; i <= nconv; ++i) {
    ConvSpec v;
    const int bi = 2 * i;  // body index of the conv; PReLU is body[2i+1]
    v.name = "body." + std::to_string(bi);
    v.wname = v.name + ".weight";
    v.bname = v.name + ".bias";
    v.sname = "body." + std::to_string(bi + 1) + ".weight";
    v.mode = kModeConv3; v.n = c.n; v.cin = cur_c; v.cout = nf;
    v.in_buf = cur; v.in_h = c.h; v.in_w = c.w; v.in_pitch = cur_pitch; v.in_coff = 0;
    v.act = kActPRelu;
    v.out_mode = kOutNHWC;
    v.out_buf = (cur == fa) ? fb : fa;
    v.out_pitch = nf; v.out_coff = 0; v.out_h = c.h; v.out_w = c.w;
    P->add_conv(v);
    cur = v.out_buf; cur_pitch = nf; cur_c = nf;
  }
  ConvSpec L;
  const int li = 2 * (nconv + 1);
  L.name = "body." + std::to_string(li);
  L.wname = L.name + ".weight"; L.bname = L.name + ".bias";
  L.mode = kModeConv3; L.n = c.n; L.cin = nf; L.cout = cl;
  L.in_buf = cur; L.in_h = c.h; L.in_w = c.w; L.in_pitch = nf;
  L.act = kActNone;
  L.out_mode = c.out_fmt == 1 ? kOutPSNCHWF16 : kOutPSNCHWF32; L.out_buf = kBufExternalOut; L.out_h = c.h; L.out_w = c.w; L.ps_r = s;
  L.base_buf = in16; L.base_pitch = 16;
  P->add_conv(L);
  return "";
}

// ------------------------------------------------------------------ RRDBNet
std::string build_rrdb(const PlanCfgLite& c, Program* P) {
  const int s = c.scale;
  if (s != 2 && s != 4) return "RRDBNet: scale must be 2 or 4";
  const int om = final_out_mode(c.out_fmt);
  if (om < 0) return "RRDBNet: unsupported output format";
  const int nb = c.depth > 0 ? c.depth : 23;
  const int nf = 64, gc = 32, slab = nf + 4 * gc;  // 192
  const int us = (s == 2) ? 2 : 1;
  if (c.h % us || c.w % us) return "RRDBNet x2: H and W must be even (mod_scale, RealESRGANer.pre_process)";
  const int th = c.h / us, tw = c.w / us;  // trunk resolution
  if (c.out_fmt == 3 && ((th * 4) % 2 || (tw * 4) % 4)) return "RRDBNet: NV12 output needs an even height and a width divisible by 4";
  const int cin0 = 3 * us * us;
  P->in_n = c.n; P->in_c = 3; P->in_h = c.h; P->in_w = c.w;
  P->out_n = c.n; P->out_c = 3; P->out_h = th * 4; P->out_w = tw * 4;
  const int in16 = P->add_buf("in16", c.n, th, tw, 16);
  const int feat = P->add_buf("feat", c.n, th, tw, nf);
  int S[3];
  for (int i = 0; i < 3; ++i) S[i] = P->add_buf("slab" + std::to_string(i), c.n, th, tw, slab);
  const int up1 = P->add_buf("up1", c.n, th * 2, tw * 2, nf);
  const int up2 = P->add_buf("up2", c.n, th * 4, tw * 4, nf);
  const int hr = P->add_buf("hr", c.n, th * 4, tw * 4, nf);
  const int hr2 = P->add_buf("hr2", c.n, th * 4, tw * 4, nf);

  PrepSpec pp;
  pp.in_fmt = c.in_fmt; pp.c = 3; pp.h = c.h; pp.w = c.w; pp.n = c.n; pp.unshuffle = us; pp.out_buf = in16;
  P->add_prep(pp);

  auto base_conv = [&](const std::string& nm, int in_buf, int ih, int iw, int ipitch, int cin, int cout) {
    ConvSpec v;
    v.name = nm; v.wname = nm + ".weight"; v.bname = nm + ".bias";
    v.mode = kModeConv3; v.n = c.n; v.cin = cin; v.cout = cout;
    v.in_buf = in_buf; v.in_h = ih; v.in_w = iw; v.in_pitch = ipitch; v.in_coff = 0;
    v.out_mode = kOutNHWC; v.out_h = ih; v.out_w = iw;
    return v;
  };
  // conv_first twice: once into the trunk-skip buffer, once as x of the first RDB (slab0[0:64))
  {
    ConvSpec v = base_conv("conv_first", in16, th, tw, 16, cin0, nf);
    v.out_buf = feat; v.out_pitch = nf;
    P->add_conv(v);
    ConvSpec u = v;
    u.out_buf = S[0]; u.out_pitch = slab;
    P->add_conv(u);
    P->flops -= u.flops();  // the duplicate is not algorithmic work
  }
  // L2 eviction priorities of the dense block (DESIGN.md section 4.4): the slab x|x1..x4 is re-read by every later
  // conv of the block and dead after conv5.  Four digits: conv1-4 loads, conv1-4 stores, conv5 loads, conv5 stores
  // (0 normal, 1 evict_last, 2 evict_first).
  int hint[4] = {1, 1, 2, 1};
  if (const char* e = getenv("SS4K_L2_HINTS")) {
    for (int i = 0; i < 4 && e[i] >= '0' && e[i] <= '2'; ++i) hint[i] = e[i] - '0';
  }
  // dead-slab discard (conv_stream.cu): on unless SS4K_DISCARD=0
  const bool use_discard = getenv("SS4K_DISCARD") == nullptr || atoi(getenv("SS4K_DISCARD")) != 0;
  for (int b = 0; b < nb; ++b) {
    for (int r = 0; r < 3; ++r) {
      const int cur = S[r], nxt = S[(r + 1) % 3];
      const std::string pre = "body." + std::to_string(b) + ".rdb" + std::to_string(r + 1) + ".conv";
      for (int k = 1; k <= 4; ++k) {
        ConvSpec v = base_conv(pre + std::to_string(k), cur, th, tw, slab, nf + (k - 1) * gc, gc);
        v.act = kActPRelu; v.const_slope = 0.2f;
        v.out_buf = cur; v.out_pitch = slab; v.out_coff = nf + (k - 1) * gc;
        v.l2_in = hint[0]; v.l2_out = hint[1];
        if (k >= 2) v.old_cin = nf + (k - 2) * gc;   // everything but conv(k-1)'s growth channels
        if (k == 1 && (b > 0 || r > 0) && use_discard) {
          // the previous block's slab is dead after its conv5 (its x stays alive when it is the RRDB input, slab 0)
          const int prev = (r + 2) % 3;
          v.discard_buf = S[prev]; v.discard_mask = prev == 0 ? 6 : 7;
          v.discard_pitch = slab; v.discard_npx = static_cast<long long>(c.n) * th * tw;
        }
        P->add_conv(v);
      }
      ConvSpec v = base_conv(pre + "5", cur, th, tw, slab, slab, nf);
      v.out_buf = nxt; v.out_pitch = slab; v.out_coff = 0;
      v.l2_in = hint[2]; v.l2_out = hint[3];
      v.old_cin = nf + 3 * gc;
      v.res1_buf = cur; v.res1_pitch = slab; v.res1_coff = 0;
      if (r < 2) {
        v.alpha = 0.2f; v.beta1 = 1.f;                    // x5*0.2 + x
      } else {
        v.alpha = 0.04f; v.beta1 = 0.2f;                  // (x5*0.2 + x)*0.2 + x_rrdb
        v.res2_buf = S[0]; v.res2_pitch = slab; v.res2_coff = 0; v.beta2 = 1.f;
      }
      P->add_conv(v);
    }
  }
  // F.interpolate(nearest, x2) is fused into the STORE of the conv in front of each upsample stage: the epilogue
  // writes every pixel 2x2 times (four TMA stores of the same tile), so conv_up1 / conv_up2 are plain 3x3 convs on
  // the upsampled grid through the row-streaming kernel.
  {  // feat + conv_body(body(feat)), stored nearest-x2 upsampled
    ConvSpec v = base_conv("conv_body", S[0], th, tw, slab, nf, nf);
    v.out_buf = up1; v.out_pitch = nf; v.up2_store = 1;
    v.res1_buf = feat; v.res1_pitch = nf; v.beta1 = 1.f;
    P->add_conv(v);
  }
  {
    ConvSpec v = base_conv("conv_up1", up1, th * 2, tw * 2, nf, nf, nf);
    v.act = kActPRelu; v.const_slope = 0.2f;
    v.out_buf = up2; v.out_pitch = nf; v.up2_store = 1;
    P->add_conv(v);
    ConvSpec u = base_conv("conv_up2", up2, th * 4, tw * 4, nf, nf, nf);
    u.act = kActPRelu; u.const_slope = 0.2f;
    u.out_buf = hr; u.out_pitch = nf;
    P->add_conv(u);
  }
  {
    ConvSpec v = base_conv("conv_hr", hr, th * 4, tw * 4, nf, nf, nf);
    v.act = kActPRelu; v.const_slope = 0.2f;
    v.out_buf = hr2; v.out_pitch = nf;
    P->add_conv(v);
    // (NV12: the epilogue converts the uint8 RGB result itself on the streaming kernel; the engine falls back to a uint8
    //  frame of its own + the rgb_to_nv12 kernel where this conv runs elsewhere)
    ConvSpec l = base_conv("conv_last", hr2, th * 4, tw * 4, nf, nf, 3);
    l.out_mode = om; l.out_buf = kBufExternalOut;
    P->add_conv(l);
  }
  return "";
}

void js_kv(std::ostringstream& o, const char* k, double v, bool last = false) {
  o << "\"" << k << "\":" << v << (last ? "" : ",");
}
void js_ks(std::ostringstream& o, const char* k, const std::string& v, bool last = false) {
  o << "\"" << k << "\":\"" << v << "\"" << (last ? "" : ",");
}

}  // namespace

std::string build_bsvd_clip(const PlanCfgLite& c, Program* P);  // bsvd_program.cpp

std::string nv12_out_check(const PlanCfgLite& cfg) {
  if (cfg.out_fmt != 3) return "";
  if (cfg.arch == 0) return "NV12 output is for RRDBNet plans: SRVGG's output feeds the colour-match glue (float / half NCHW)";
  if (cfg.arch == 2) return "NV12 output is for RRDBNet plans: BSVD's output feeds the sharpen glue (float / half NCHW)";
  if (cfg.arch != 1) return "";
  const long long oh = static_cast<long long>(cfg.h) * cfg.scale, ow = static_cast<long long>(cfg.w) * cfg.scale;
  if (oh % 2 || ow % 4) return "NV12 output needs an even output height and an output width divisible by 4";
  return "";
}

std::string build_program(const PlanCfgLite& cfg, Program* out) {
  out->in_fmt = cfg.in_fmt;
  out->out_fmt = cfg.out_fmt;
  if (cfg.n < 1 || cfg.h < 1 || cfg.w < 1) return "bad frame geometry";
  {
    const std::string e = nv12_out_check(cfg);
    if (!e.empty()) return e;
  }
  switch (cfg.arch) {
    case 0: return build_srvgg(cfg, out);
    case 1: return build_rrdb(cfg, out);
    case 2: return build_bsvd_clip(cfg, out);
    default: return "unknown arch";
  }
}

std::string Program::to_json() const {
  std::ostringstream o;
  o.precision(9);
  o << "{";
  js_kv(o, "in_n", in_n); js_kv(o, "in_c", in_c); js_kv(o, "in_h", in_h); js_kv(o, "in_w", in_w);
  js_kv(o, "out_n", out_n); js_kv(o, "out_c", out_c); js_kv(o, "out_h", out_h); js_kv(o, "out_w", out_w);
  js_kv(o, "in_fmt", in_fmt); js_kv(o, "out_fmt", out_fmt); js_kv(o, "flops", flops);
  o << "\"bufs\":[";
  for (size_t i = 0; i < bufs.size(); ++i) {
    const BufSpec& b = bufs[i];
    o << "{";
    js_ks(o, "name", b.name); js_kv(o, "n", b.n); js_kv(o, "h", b.h); js_kv(o, "w", b.w);
    js_kv(o, "zero", b.zero_init ? 1 : 0);
    js_kv(o, "pitch", b.pitch, true);
    o << "}" << (i + 1 < bufs.size() ? "," : "");
  }
  o << "],\"steps\":[";
  for (size_t i = 0; i < steps.size(); ++i) {
    const Step& s = steps[i];
    o << "{";
    if (s.kind == 0) {
      const PrepSpec& p = s.prep;
      js_ks(o, "kind", "prep"); js_kv(o, "in_fmt", p.in_fmt); js_kv(o, "c", p.c); js_kv(o, "h", p.h);
      js_kv(o, "w", p.w); js_kv(o, "n", p.n); js_kv(o, "n0", p.n0); js_kv(o, "unshuffle", p.unshuffle);
      js_kv(o, "out_buf", p.out_buf); js_kv(o, "out_lo_buf", p.out_lo_buf);
      js_kv(o, "fill_ch", p.fill_ch); js_kv(o, "fill_val", p.fill_val, true);
    } else if (s.kind == 2) {
      js_ks(o, "kind", "rgb_to_nv12", true);
    } else {
      const ConvSpec& c = s.conv;
      js_ks(o, "kind", "conv"); js_ks(o, "name", c.name); js_ks(o, "wname", c.wname);
      js_ks(o, "bname", c.bname); js_ks(o, "sname", c.sname); js_kv(o, "const_slope", c.const_slope);
      js_kv(o, "mode", c.mode); js_kv(o, "n", c.n); js_kv(o, "n0", c.n0); js_kv(o, "n_total", c.n_total); js_kv(o, "cin", c.cin); js_kv(o, "cout", c.cout);
      js_kv(o, "in_buf", c.in_buf); js_kv(o, "in_lo_buf", c.in_lo_buf); js_kv(o, "in_h", c.in_h);
      js_kv(o, "in_w", c.in_w); js_kv(o, "in_pitch", c.in_pitch); js_kv(o, "in_coff", c.in_coff);
      js_kv(o, "act", c.act); js_kv(o, "alpha", c.alpha); js_kv(o, "beta1", c.beta1);
      js_kv(o, "beta2", c.beta2); js_kv(o, "res1_buf", c.res1_buf); js_kv(o, "res1_lo_buf", c.res1_lo_buf); js_kv(o, "res2_lo_buf", c.res2_lo_buf); js_kv(o, "res1_pitch", c.res1_pitch);
      js_kv(o, "res1_coff", c.res1_coff); js_kv(o, "res2_buf", c.res2_buf);
      js_kv(o, "res2_pitch", c.res2_pitch); js_kv(o, "res2_coff", c.res2_coff);
      js_kv(o, "out_mode", c.out_mode); js_kv(o, "out_buf", c.out_buf); js_kv(o, "out_lo_buf", c.out_lo_buf);
      js_kv(o, "out2_buf", c.out2_buf); js_kv(o, "out3_buf", c.out3_buf); js_kv(o, "out_pitch", c.out_pitch);
      js_kv(o, "out_coff", c.out_coff); js_kv(o, "out_h", c.out_h); js_kv(o, "out_w", c.out_w);
      js_kv(o, "ps_r", c.ps_r); js_kv(o, "fold", c.fold); js_kv(o, "round_u8", c.round_u8);
      js_kv(o, "base_buf", c.base_buf); js_kv(o, "base_pitch", c.base_pitch); js_kv(o, "wperm", c.wperm);
      js_kv(o, "neg_first", c.neg_first); js_kv(o, "res1_nch", c.res1_nch); js_kv(o, "tshift", c.tshift);
      js_kv(o, "up2_store", c.up2_store);
      js_kv(o, "old_cin", c.old_cin); js_kv(o, "l2_in", c.l2_in); js_kv(o, "l2_out", c.l2_out);
      js_kv(o, "discard_buf", c.discard_buf); js_kv(o, "discard_mask", c.discard_mask);
      js_kv(o, "split", c.split, true);
    }
    o << "}" << (i + 1 < steps.size() ? "," : "");
  }
  o << "]}";
  return o.str();
}

}  // namespace ss4k
