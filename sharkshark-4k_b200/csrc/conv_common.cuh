// Device-side helpers shared by the tcgen05 convolution kernels (conv_tc.cu, conv_stream.cu):
// PTX wrappers (mbarrier, TMA, tcgen05), 16-bit pack/unpack and the fused epilogue
// (bias / PReLU / ReLU6 / scaled residual adds / NHWC, PixelShuffle, NCHW, uint8, temporal-shift stores).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv_params.h"

namespace ss4k {
namespace {

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a pipeline bug must not hang the GPU.  After ~4 s the kernel records where it
// was stuck and traps (the host then reports SS4K_E_CUDA with the diagnostic).
__device__ __noinline__ void mbar_timeout(int32_t* err, int tag, uint32_t parity) {
  if (err != nullptr) {
    err[0] = tag;
    err[1] = static_cast<int32_t>(blockIdx.x);
    err[2] = static_cast<int32_t>(threadIdx.x);
    err[3] = static_cast<int32_t>(parity);
    __threadfence_system();
  }
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int32_t* err, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (globaltimer_ns() - t0 > 4000000000ull) mbar_timeout(err, tag, parity);
  }
}

// Wait with the retry loop INSIDE the asm block: the surrounding C++ control flow stays warp-uniform for
// ptxas, so descriptors / addresses of the MMA and TMA issue loops live in uniform registers.
// Bounded: after ~4 s without progress the kernel traps (a pipeline bug must not hang the GPU).
__device__ __forceinline__ void mbar_wait_u(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1, P2;\n\t"
      ".reg .u64 t0, t1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra LAB_DONE;\n\t"
      "mov.u64 t0, %%globaltimer;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra LAB_DONE;\n\t"
      "mov.u64 t1, %%globaltimer;\n\t"
      "sub.u64 t1, t1, t0;\n\t"
      "setp.lt.u64 P2, t1, 4000000000;\n\t"
      "@P2 bra LAB_WAIT;\n\t"
      "trap;\n\t"
      "LAB_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
      : "memory");
}
// L2 eviction-priority policy for TMA loads / stores: 0 evict_normal, 1 evict_last, 2 evict_first
__device__ __forceinline__ uint64_t l2_policy(int kind) {
  uint64_t p;
  if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_5d_hint(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                                 int c0, int c1, int c2, int c3, int c4, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], M=128, K=16, 16-bit operands, fp32 accumulate
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// whole-warp (convergent) variants: every lane executes the statement, one elected lane issues
__device__ __forceinline__ void umma_f16_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Same, with the 64-bit shared-memory descriptors given as their low words (start address >> 4); the high word
// (SBO = 1024 B, version 1, swizzle 128B) is a constant.  Keeps the per-MMA issue cost at a couple of uniform adds.
__device__ __forceinline__ void umma_f16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, e;\n\t"
      ".reg .b64 da, db;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}"
      :
      : "r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(0x40004040u)
      : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16p(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// registers -> TMEM: 16 consecutive fp32 columns of this warp's 32 lanes (lane i writes row i)
__device__ __forceinline__ void tmem_st16p(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void lds128(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}

// K-major, swizzle-128B shared memory matrix descriptor (sm_100 "version 1"):
//   rows are 128 bytes (64 x 16-bit), 8-row groups are 1024 bytes apart (SBO), LBO unused.
//   base_offset = row phase of the start address inside the 1024-byte swizzle pattern.
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr, uint32_t base_offset) {
  return static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(1024u >> 4) << 32) |
         (1ull << 46) | (static_cast<uint64_t>(base_offset & 7u) << 49) | (2ull << 61);
}

// ---------------------------------------------------------------- 16-bit pack / unpack
__device__ __forceinline__ uint32_t pack2(float a, float b, bool bf16) {
  if (bf16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack2(uint32_t u, bool bf16) {
  if (bf16) {
    __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&u);
    return __bfloat1622float2(h);
  }
  __half2 h = *reinterpret_cast<__half2*>(&u);
  return __half22float2(h);
}
__device__ __forceinline__ float round16(float a, bool bf16) {
  return bf16 ? __bfloat162float(__float2bfloat16_rn(a)) : __half2float(__float2half_rn(a));
}

__device__ __forceinline__ void add_residual16(float (&v)[16], const void* res, size_t elem_off,
                                               float beta, bool bf16) {
  const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(res) + elem_off);
  // plain (coherent) loads: the RRDB tail conv updates its residual buffer in place
  const uint4 q0 = *p;
  const uint4 q1 = *(p + 1);
  const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float2 f = unpack2(w[i], bf16);
    v[2 * i] = fmaf(beta, f.x, v[2 * i]);
    v[2 * i + 1] = fmaf(beta, f.y, v[2 * i + 1]);
  }
}

__device__ __forceinline__ void store8(void* base, size_t elem_off, const float* v, bool bf16) {
  uint4 q;
  q.x = pack2(v[0], v[1], bf16);
  q.y = pack2(v[2], v[3], bf16);
  q.z = pack2(v[4], v[5], bf16);
  q.w = pack2(v[6], v[7], bf16);
  *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(base) + elem_off) = q;
}
__device__ __forceinline__ void store8_lo(void* base, size_t elem_off, const float* v, bool bf16) {
  float r[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = v[i] - round16(v[i], bf16);
  store8(base, elem_off, r, bf16);
}

// Where one output image of a launch lives: its image index in the output and residual tensors (relative to their base
// pointers), its frame index in the clip (temporal-shift boundary guards) and the distances, in frames, to the
// neighbouring frames' images (E.off_prev / E.off_next are one frame each).  They all follow from the launch's image
// index n, except where a tensor is a ring of frames that wraps inside the launch (BSVD streams, conv_stream.cu::ring_img).
struct ImgAt {
  int out, res1, res2, t, prev, next;
};
__device__ __forceinline__ ImgAt img_at(const Epilogue& E, int n) { return ImgAt{n, n, n, E.t0 + n, 1, 1}; }

// One 16-channel chunk of one output pixel: bias, activation, residuals, store.
//   ch0: channel index of v[0] within the conv's (padded) output channels
//   (ay, ax): pixel in A space; sub: accumulator phase (kModeUp2)
__device__ __forceinline__ void epilogue_chunk(const Epilogue& E, int mode, const ImgAt& I, int ay, int ax, int sub,
                                               int ch0, float (&v)[16]) {
  const int n = I.out;
  const bool bf16 = E.is_bf16 != 0;
  // ---- bias + activation
  {
    if (E.bias != nullptr) {  // null: the bias was already added by the accumulator-init MMA (conv_stream.cu)
      const float4* bp = reinterpret_cast<const float4*>(E.bias + ch0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b = __ldg(bp + q);
        v[4 * q + 0] += b.x;
        v[4 * q + 1] += b.y;
        v[4 * q + 2] += b.z;
        v[4 * q + 3] += b.w;
      }
    }
    if (E.act == kActPRelu && E.slope == nullptr) {
      const float sl = E.slope_const;
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = v[i] >= 0.f ? v[i] : v[i] * sl;
    } else if (E.act == kActPRelu) {
      const float4* sp = reinterpret_cast<const float4*>(E.slope + ch0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 s = __ldg(sp + q);
        v[4 * q + 0] = v[4 * q + 0] >= 0.f ? v[4 * q + 0] : v[4 * q + 0] * s.x;
        v[4 * q + 1] = v[4 * q + 1] >= 0.f ? v[4 * q + 1] : v[4 * q + 1] * s.y;
        v[4 * q + 2] = v[4 * q + 2] >= 0.f ? v[4 * q + 2] : v[4 * q + 2] * s.z;
        v[4 * q + 3] = v[4 * q + 3] >= 0.f ? v[4 * q + 3] : v[4 * q + 3] * s.w;
      }
    } else if (E.act == kActRelu6) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = fminf(fmaxf(v[i], 0.f), 6.f);
    }
    if (E.alpha != 1.0f) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] *= E.alpha;
    }
  }
  // ---- output pixel / channel
  int oy = ay, ox = ax, oc = ch0;
  if (mode == kModeUp2) {
    oy = 2 * ay + (sub >> 1);
    ox = 2 * ax + (sub & 1);
  }
  if (E.out_mode == kOutPS2NHWC) {
    const int cq = E.cout >> 2;  // channels of the shuffled output
    const int ab = ch0 / cq;
    oc = ch0 - ab * cq;
    oy = 2 * oy + (ab >> 1);
    ox = 2 * ox + (ab & 1);
  }
  const size_t pix = (static_cast<size_t>(n) * E.out_h + oy) * E.out_w + ox;
  // ---- residuals (indexed at the output pixel, NHWC)
  if (E.res1 != nullptr) {
    const size_t p1 = (static_cast<size_t>(I.res1) * E.out_h + oy) * E.out_w + ox;
    if (E.res1_nch > 0) {
      if (oc < E.res1_nch) {
        float r[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = 0.f;
        add_residual16(r, E.res1, p1 * E.res1_pitch + E.res1_coff + oc, E.beta1, bf16);
        if (E.res1_lo_off != 0) add_residual16(r, E.res1, p1 * E.res1_pitch + E.res1_coff + oc + E.res1_lo_off, E.beta1, bf16);
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (oc + i < E.res1_nch) v[i] += r[i];
      }
    } else {
      add_residual16(v, E.res1, p1 * E.res1_pitch + E.res1_coff + oc, E.beta1, bf16);
      if (E.res1_lo_off != 0) add_residual16(v, E.res1, p1 * E.res1_pitch + E.res1_coff + oc + E.res1_lo_off, E.beta1, bf16);
    }
  }
  if (E.res2 != nullptr) {
    const size_t p2 = (static_cast<size_t>(I.res2) * E.out_h + oy) * E.out_w + ox;
    add_residual16(v, E.res2, p2 * E.res2_pitch + E.res2_coff + oc, E.beta2, bf16);
    if (E.res2_lo_off != 0) add_residual16(v, E.res2, p2 * E.res2_pitch + E.res2_coff + oc + E.res2_lo_off, E.beta2, bf16);
  }
  // ---- store
  switch (E.out_mode) {
    case kOutNHWC:
    case kOutPS2NHWC: {
      const size_t off = pix * E.out_pitch + E.out_coff + oc;
      if (E.fold > 0) {  // temporal-shift scatter
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c = oc + 8 * h;
          const int t = I.t;
          int64_t delta = 0;
          bool ok = true;
          if (c < E.fold) { delta = E.off_prev * I.prev; ok = t > 0; }
          else if (c < 2 * E.fold) { delta = E.off_next * I.next; ok = t < E.t_count - 1; }
          if (ok) {
            const size_t o2 = static_cast<size_t>(static_cast<int64_t>(off) + 8 * h + delta);
            store8(E.out, o2, v + 8 * h, bf16);
            if (E.out_lo != nullptr) store8_lo(E.out_lo, o2, v + 8 * h, bf16);
          }
        }
      } else if (E.up2_store) {  // nearest-x2 upsample fused into the store (RRDBNet upsample stages)
#pragma unroll
        for (int ab = 0; ab < 4; ++ab) {
          const size_t p2 = (static_cast<size_t>(n) * 2 * E.out_h + 2 * oy + (ab >> 1)) * (2 * E.out_w) + 2 * ox + (ab & 1);
          const size_t o2 = p2 * E.out_pitch + E.out_coff + oc;
          store8(E.out, o2, v, bf16);
          store8(E.out, o2 + 8, v + 8, bf16);
        }
      } else {
        store8(E.out, off, v, bf16);
        store8(E.out, off + 8, v + 8, bf16);
        if (E.out_lo != nullptr) {
          store8_lo(E.out_lo, off, v, bf16);
          store8_lo(E.out_lo, off + 8, v + 8, bf16);
        }
      }
    } break;
    case kOutScatterNHWC: {
      const size_t off = pix * E.out_pitch + E.out_coff + oc;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = oc + 8 * h;
        void* dst = c < E.fold ? E.out2 : (c < 2 * E.fold ? E.out3 : E.out);
        store8(dst, off + 8 * h, v + 8 * h, bf16);
      }
    } break;
    case kOutNCHWF32: {
      float* o = reinterpret_cast<float*>(E.out);
      const size_t plane = static_cast<size_t>(E.out_h) * E.out_w;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int c = oc + i;
        if (c < E.cout) o[(static_cast<size_t>(n) * E.cout + c) * plane + static_cast<size_t>(oy) * E.out_w + ox] = v[i];
      }
    } break;
    case kOutNCHWF16: {
      __half* o = reinterpret_cast<__half*>(E.out);
      const size_t plane = static_cast<size_t>(E.out_h) * E.out_w;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int c = oc + i;
        if (c < E.cout)
          o[(static_cast<size_t>(n) * E.cout + c) * plane + static_cast<size_t>(oy) * E.out_w + ox] = __float2half_rn(v[i]);
      }
    } break;
    case kOutU8NHWC: {
      uint8_t* o = reinterpret_cast<uint8_t*>(E.out) + pix * E.cout;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int c = oc + i;
        if (c < E.cout) {
          float f = fminf(fmaxf(v[i], 0.f), 1.f) * 255.f;
          if (E.round_u8) f = rintf(f);
          o[c] = static_cast<uint8_t>(f);
        }
      }
    } break;
    case kOutPSNCHWF16:
    case kOutPSNCHWF32: {
      // conv channel ch = c*r*r + a*r + b  ->  out[n, c, oy*r + a, ox*r + b]  (+ base[n, oy, ox, c])
      float* o = reinterpret_cast<float*>(E.out);
      const int r = E.ps_r, rr = r * r;
      const int oc_total = E.cout / rr;
      const int OH = E.out_h * r, OW = E.out_w * r;
      const uint16_t* bpix = E.base != nullptr
                                 ? reinterpret_cast<const uint16_t*>(E.base) + pix * E.base_pitch
                                 : nullptr;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int ch = oc + i;
        if (ch < E.cout) {
          const int c = ch / rr, rem = ch - c * rr;
          const int a = rem / r, b = rem - a * r;
          float val = v[i];
          if (bpix != nullptr) {
            const uint16_t raw = __ldg(bpix + c);
            val += bf16 ? __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&raw))
                        : __half2float(*reinterpret_cast<const __half*>(&raw));
          }
          const size_t oi = ((static_cast<size_t>(n) * oc_total + c) * OH + (static_cast<size_t>(oy) * r + a)) * OW + static_cast<size_t>(ox) * r + b;
          if (E.out_mode == kOutPSNCHWF16) reinterpret_cast<__half*>(E.out)[oi] = __float2half_rn(val);
          else o[oi] = val;
        }
      }
    } break;
    default:
      break;
  }
}


}  // namespace
}  // namespace ss4k
