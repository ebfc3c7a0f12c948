// tcgen05 / TMEM / TMA implicit-GEMM 3x3 convolution for sm_100a.
//
// Replaces torch.nn.Conv2d(k=3) -> cuDNN/TensorRT on the reference's hot path
// (src/upscale/model/realesrgan/factory.py:44-67 SRVGG convs, basicsr RRDBNet convs reached from
//  factory.py:113-125, src/upscale/model/bsvd/model.py:22-53,231-323 BSVD convs).
//
// Design (DESIGN.md section 4):
//   * activations NHWC 16-bit in HBM; GEMM M = 128 consecutive pixels of one image row (TMEM lanes),
//     N = output channels (TMEM columns), K = 9 taps x input channels in 64-channel blocks.
//   * one persistent CTA per SM; a tile is R output rows x 128 pixels with R accumulators in TMEM,
//     double buffered (2 x 256 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
//   * each input halo row (130 pixels x 64 channels = one swizzle-128B K-major slab) is loaded ONCE by
//     TMA (zero fill outside the image == conv padding) and consumed by up to 9 tap-MMAs: the 3
//     horizontal taps are the same slab addressed with a 0/1/2-row shifted start address, the 3
//     vertical taps feed 3 different accumulators.  No im2col, no 9x re-read of activations.
//   * weights for a whole 64-channel K block (all taps) stay in shared memory, double buffered
//     (or resident for the whole kernel when K fits one block).
//   * warp 0 = TMA producer, warp 1 = MMA issuer (one elected thread), warps 2..5 = epilogue
//     (TMEM -> registers -> bias / PReLU / ReLU6 / scaled residual adds -> 16-byte NHWC stores,
//      or PixelShuffle / NCHW / uint8 / temporal-shift scatter stores).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv_common.cuh"
#include "conv_params.h"

namespace ss4k {

// ---------------------------------------------------------------- the kernel
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_tcgen05_kernel(const __grid_constant__ ConvParams P) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = smem_base;
  const uint32_t a_base = w_base + static_cast<uint32_t>(P.w_slots) * P.w_slot_bytes;
  const uint32_t bar_base = a_base + static_cast<uint32_t>(P.a_slots) * P.a_slot_bytes;
  // barrier map (8 bytes each)
  const uint32_t a_full = bar_base;                   // [kMaxASlots]
  const uint32_t a_empty = bar_base + 8 * kMaxASlots; // [kMaxASlots]
  const uint32_t w_full = bar_base + 16 * kMaxASlots; // [2]
  const uint32_t w_empty = w_full + 16;               // [2]
  const uint32_t t_full = w_empty + 16;               // [2]
  const uint32_t t_empty = t_full + 16;               // [2]
  const uint32_t tmem_slot = t_empty + 16;            // uint32
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&P.tmA[0]);
    prefetch_tmap(&P.tmW);
    for (int i = 0; i < kMaxASlots; ++i) {
      mbar_init(a_full + 8 * i, 1);
      mbar_init(a_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(w_full + 8 * i, 1);
      mbar_init(w_empty + 8 * i, 1);
      mbar_init(t_full + 8 * i, 1);
      mbar_init(t_empty + 8 * i, 4);  // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int in_rows = P.R + P.max_dr;
  const int tiles_per_img = P.tiles_y * P.tiles_x * P.n_chunks;

  if (warp == 0) {
    // ======================================================= TMA producer
    if (lane == 0) {
      uint32_t as = 0, aph = 0, ws = 0, wph = 0;
      bool w_loaded = false;
      for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
        const int n = tile / tiles_per_img;
        int rem = tile - n * tiles_per_img;
        const int ty = rem / (P.tiles_x * P.n_chunks);
        rem -= ty * (P.tiles_x * P.n_chunks);
        const int tx = rem / P.n_chunks;
        const int nc = rem - tx * P.n_chunks;
        const int y0 = ty * P.R, x0 = tx * kTileW;
        for (int kbi = 0; kbi < P.nkb; ++kbi) {
          if (!(P.w_resident && w_loaded)) {
            mbar_wait(w_empty + 8 * ws, wph ^ 1, P.err, 1);
            if (P.dbg_flags & 2) {
              mbar_arrive(w_full + 8 * ws);
            } else {
              mbar_expect_tx(w_full + 8 * ws, P.w_tx);
              tma_load_3d(w_base + ws * P.w_slot_bytes, &P.tmW, w_full + 8 * ws, 0, nc * P.n_cta,
                          kbi * P.ntaps);
            }
            w_loaded = true;
            if (++ws == static_cast<uint32_t>(P.w_slots)) { ws = 0; wph ^= 1; }
          }
          const KBlock kb = P.kb[kbi];
          const CUtensorMap* tm = &P.tmA[kb.tmap];
          for (int r = 0; r < in_rows; ++r) {
            mbar_wait(a_empty + 8 * as, aph ^ 1, P.err, 2);
            if (P.dbg_flags & 2) {
              mbar_arrive(a_full + 8 * as);
              if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
              continue;
            }
            mbar_expect_tx(a_full + 8 * as, P.a_row_tx);
            const uint32_t dst = a_base + as * P.a_slot_bytes;
            const int y = y0 - 1 + r;
            if (P.desc_mode == 2) {
#pragma unroll
              for (int s = 0; s < 3; ++s)
                tma_load_5d(dst + s * P.a_sub_bytes, tm, a_full + 8 * as, kb.c0, x0 - 1 + s, kb.p, y, n + P.n_in0);
            } else {
              tma_load_5d(dst, tm, a_full + 8 * as, kb.c0, x0 - 1, kb.p, y, n + P.n_in0);
            }
            if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ======================================================= MMA issuer
    if (lane == 0) {
      uint32_t as = 0, aph = 0, ws = 0, wph = 0;
      bool w_ready = false;
      uint32_t wcur = w_base;
      int it = 0;
      for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
        const uint32_t ts = it & 1, tph = (it >> 1) & 1;
        mbar_wait(t_empty + 8 * ts, tph ^ 1, P.err, 3);
        tcgen05_after_sync();
        const uint32_t tacc = tmem_base + ts * kAccStageCols;
        uint32_t started = 0;
        for (int kbi = 0; kbi < P.nkb; ++kbi) {
          uint32_t this_ws = ws;
          if (!(P.w_resident && w_ready)) {
            mbar_wait(w_full + 8 * ws, wph, P.err, 4);
            tcgen05_after_sync();
            wcur = w_base + ws * P.w_slot_bytes;
            w_ready = true;
            this_ws = ws;
            if (++ws == static_cast<uint32_t>(P.w_slots)) { ws = 0; wph ^= 1; }
          }
          for (int r = 0; r < in_rows; ++r) {
            mbar_wait(a_full + 8 * as, aph, P.err, 5);
            tcgen05_after_sync();
            const uint32_t arow = a_base + as * P.a_slot_bytes;
            for (int t = 0; t < P.ntaps && !(P.dbg_flags & 1); ++t) {
              const Tap tap = P.taps[t];
              const int j = r - tap.dr;
              if (j < 0 || j >= P.R) continue;
              const uint32_t mask = P.ksmask[kbi][t];
              if (mask == 0) continue;
              const uint32_t acc = static_cast<uint32_t>(j * P.nsub + tap.sub);
              const uint32_t d_tmem = tacc + acc * P.acc_stride;
              uint32_t a_addr, boff;
              if (P.desc_mode == 2) {
                a_addr = arow + tap.shift * P.a_sub_bytes;
                boff = 0;
              } else {
                a_addr = arow + tap.shift * kRowBytes;
                boff = P.desc_mode == 1 ? static_cast<uint32_t>(tap.shift) : 0u;
              }
              const uint32_t b_addr = wcur + t * P.w_tile_bytes;
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                if (mask & (1u << ks)) {
                  umma_f16(d_tmem, make_sdesc(a_addr + ks * 32, boff), make_sdesc(b_addr + ks * 32, 0),
                           P.idesc, (started >> acc) & 1u);
                  started |= 1u << acc;
                }
              }
            }
            umma_commit(a_empty + 8 * as);  // slot reusable once these MMAs have read it
            if (++as == static_cast<uint32_t>(P.a_slots)) { as = 0; aph ^= 1; }
          }
          if (!P.w_resident) umma_commit(w_empty + 8 * this_ws);
        }
        umma_commit(t_full + 8 * ts);  // accumulators of this tile complete
      }
    }
  } else {
    // ======================================================= epilogue (warps 2..5)
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int m = q * 32 + lane;       // accumulator row == pixel inside the tile row
    const int nacc = P.R * P.nsub;
    int it = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
      const int n = tile / tiles_per_img;
      int rem = tile - n * tiles_per_img;
      const int ty = rem / (P.tiles_x * P.n_chunks);
      rem -= ty * (P.tiles_x * P.n_chunks);
      const int tx = rem / P.n_chunks;
      const int nc = rem - tx * P.n_chunks;
      const int y0 = ty * P.R, x0 = tx * kTileW;
      const uint32_t ts = it & 1, tph = (it >> 1) & 1;
      mbar_wait(t_full + 8 * ts, tph, P.err, 6);
      tcgen05_after_sync();
      const uint32_t tacc = tmem_base + ts * kAccStageCols + (static_cast<uint32_t>(q * 32) << 16);
      const int ax = x0 + m;
      for (int ai = 0; ai < nacc; ++ai) {
        const int j = ai / P.nsub;
        const int sub = ai - j * P.nsub;
        const int ay = y0 + j;
        if (ay >= P.H) break;  // warp-uniform
        const bool valid = ax < P.W;
        for (int cb = 0; cb < P.n_cta; cb += 16) {
          uint32_t raw[16];
          tmem_ld16(tacc + ai * P.acc_stride + cb, raw);
          tmem_ld_wait();
          if (valid && !(P.dbg_flags & 4)) {
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(raw[i]);
            epilogue_chunk(P.ep, P.mode, img_at(P.ep, n), ay, ax, sub, nc * P.n_cta + cb, v);
          }
        }
      }
      tcgen05_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + 8 * ts);
    }
  }

  // ---------------------------------------------------------------- teardown
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(static_cast<uint32_t>(kTmemCols))
                 : "memory");
  }
}

// ---------------------------------------------------------------- host launcher
cudaError_t conv_tc_prepare() {
  return cudaFuncSetAttribute(conv3x3_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              kSmemBytes);
}

cudaError_t conv_tc_launch(const ConvParams& p, int grid, cudaStream_t stream) {
  conv3x3_tcgen05_kernel<<<grid, kConvThreads, kSmemBytes, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace ss4k
