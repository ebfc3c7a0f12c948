// Service glue of the upscaler (HBM-bound elementwise / stencil / reduction kernels around the convnets).
//
// Reference: src/upscale/fsrcnn_upscaler.py
//   upscale_multi  :168-233  /255 + NHWC->NCHW (+ area downscale), model, per-(N,C) mean / unbiased-std match
//                            to the LR frame (:188-199), local colour match (area /8, 17x17 sigma-8 reflect
//                            gaussian, bilinear up, subtract :201-218), clamp, bicubic resize (:222-231),
//                            *255 -> uint8 truncating, ->NHWC (:232-233)
//   upscale_single :235-326  denoise blend: 3x3 reflect sharpen + clamp, 0.8*den + 0.2*orig (:273-281),
//                            HR sharpen (:298-299), mean/std match (:302-313)
//   blur_ker / sharpen_ker :20-84
// The reference runs ~10 separate ATen passes over the HR frame; here: one statistics pass, one pooling pass,
// a tiny low-resolution blur and ONE finalising pass that applies the affine match, subtracts the bilinearly
// upsampled colour difference, clamps and writes uint8 NHWC.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <stdint.h>

#include "../../include/ss4k.h"

namespace ss4k {
namespace {

// image access: fmt 0 float NCHW, 1 half NCHW, 2 uint8 NHWC (value / 255)
struct Img {
  const void* p;
  int fmt, N, C, H, W;
  __device__ __forceinline__ float at(int n, int c, int y, int x) const {
    if (fmt == 0) return reinterpret_cast<const float*>(p)[((static_cast<size_t>(n) * C + c) * H + y) * W + x];
    if (fmt == 1) return __half2float(reinterpret_cast<const __half*>(p)[((static_cast<size_t>(n) * C + c) * H + y) * W + x]);
    if (fmt == 3) {  // NV12 frame (Y plane + interleaved UV), BT.709 limited range, nearest chroma: same arithmetic as prep_kernel
      const uint8_t* frame = reinterpret_cast<const uint8_t*>(p) + static_cast<size_t>(n) * (static_cast<size_t>(H) * W * 3 / 2);
      const float yy = (static_cast<float>(frame[static_cast<size_t>(y) * W + x]) - 16.f) * (1.f / 219.f);
      const uint8_t* uv = frame + static_cast<size_t>(H) * W + static_cast<size_t>(y >> 1) * W + (x & ~1);
      const float cb = (static_cast<float>(uv[0]) - 128.f) * (1.f / 224.f), cr = (static_cast<float>(uv[1]) - 128.f) * (1.f / 224.f);
      const float v = c == 0 ? yy + 1.5748f * cr : (c == 1 ? yy - 0.187324f * cb - 0.468124f * cr : yy + 1.8556f * cb);
      return fminf(fmaxf(v, 0.f), 1.f);
    }
    return static_cast<float>(reinterpret_cast<const uint8_t*>(p)[((static_cast<size_t>(n) * H + y) * W + x) * C + c]) / 255.0f;
  }
};

// ---- per (n, c) sum and sum of squares (double) ----------------------------------------------------
__global__ void chan_stats_kernel(Img im, double* __restrict__ sums /* [N*C][2] */) {
  const int nc = blockIdx.y;
  const int n = nc / im.C, c = nc - n * im.C;
  const size_t total = static_cast<size_t>(im.H) * im.W;
  double s = 0.0, q = 0.0;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int y = static_cast<int>(i / im.W), x = static_cast<int>(i - static_cast<size_t>(y) * im.W);
    const float v = im.at(n, c, y, x);
    s += v;
    q += static_cast<double>(v) * v;
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  __shared__ double sh[2][32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s; sh[1][w] = q; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    s = l < nw ? sh[0][l] : 0.0;
    q = l < nw ? sh[1][l] : 0.0;
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (l == 0) {
      atomicAdd(&sums[2 * nc], s);
      atomicAdd(&sums[2 * nc + 1], q);
    }
  }
}

// half NCHW planes (the net's output): 16-byte loads, no index arithmetic -- the plane is contiguous.  Same
// accumulation type as the general kernel (every element is added in double).
__global__ void chan_stats_half_kernel(const uint4* __restrict__ img, size_t vec_per_plane, double* __restrict__ sums) {
  const int nc = blockIdx.y;
  const uint4* p = img + static_cast<size_t>(nc) * vec_per_plane;
  double s = 0.0, q = 0.0;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < vec_per_plane;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const uint4 v = __ldg(p + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
      s += f.x;
      q += static_cast<double>(f.x) * f.x;
      s += f.y;
      q += static_cast<double>(f.y) * f.y;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  __shared__ double sh[2][32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s; sh[1][w] = q; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    s = l < nw ? sh[0][l] : 0.0;
    q = l < nw ? sh[1][l] : 0.0;
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (l == 0) {
      atomicAdd(&sums[2 * nc], s);
      atomicAdd(&sums[2 * nc + 1], q);
    }
  }
}

// affine map of the distribution match: hr' = a*hr + b with a = std_lr / (std_hr + 1e-8), b = mean_lr - a*mean_hr
// (unbiased std like torch.Tensor.std)
__device__ __forceinline__ void match_coeffs(const double* hr_sums, const double* lr_sums, int nc, double cnt_hr,
                                             double cnt_lr, float* a, float* b) {
  if (hr_sums == nullptr) { *a = 1.f; *b = 0.f; return; }
  const double mh = hr_sums[2 * nc] / cnt_hr, ml = lr_sums[2 * nc] / cnt_lr;
  double vh = (hr_sums[2 * nc + 1] - cnt_hr * mh * mh) / (cnt_hr - 1.0);
  double vl = (lr_sums[2 * nc + 1] - cnt_lr * ml * ml) / (cnt_lr - 1.0);
  vh = vh > 0.0 ? vh : 0.0;
  vl = vl > 0.0 ? vl : 0.0;
  const double aa = sqrt(vl) / (sqrt(vh) + 1e-8);
  *a = static_cast<float>(aa);
  *b = static_cast<float>(ml - aa * mh);
}

// ---- F.interpolate(mode='area') == adaptive average pooling -> float NCHW ---------------------------
__global__ void area_pool_kernel(Img im, float* __restrict__ out, int oh, int ow) {
  const size_t total = static_cast<size_t>(im.N) * im.C * oh * ow;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ox = static_cast<int>(idx % ow);
  const int oy = static_cast<int>((idx / ow) % oh);
  const int c = static_cast<int>((idx / (static_cast<size_t>(ow) * oh)) % im.C);
  const int n = static_cast<int>(idx / (static_cast<size_t>(ow) * oh * im.C));
  const int y0 = static_cast<int>((static_cast<int64_t>(oy) * im.H) / oh);
  const int y1 = static_cast<int>((static_cast<int64_t>(oy + 1) * im.H + oh - 1) / oh);
  const int x0 = static_cast<int>((static_cast<int64_t>(ox) * im.W) / ow);
  const int x1 = static_cast<int>((static_cast<int64_t>(ox + 1) * im.W + ow - 1) / ow);
  float s = 0.f;
  for (int y = y0; y < y1; ++y)
    for (int x = x0; x < x1; ++x) s += im.at(n, c, y, x);
  out[idx] = s / static_cast<float>((y1 - y0) * (x1 - x0));
}

__device__ __forceinline__ int reflect(int i, int n) {  // padding_mode='reflect' (no edge repeat)
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return i;
}

// ---- low-resolution colour difference: blur_k(a*hb + b - lb), k x k normalised gaussian, reflect padding ----
__global__ void blur_diff_kernel(const float* __restrict__ hb, const float* __restrict__ lb, float* __restrict__ diff,
                                 const float* __restrict__ kern, int ksize, int N, int C, int h, int w,
                                 const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr) {
  const size_t total = static_cast<size_t>(N) * C * h * w;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int x = static_cast<int>(idx % w);
  const int y = static_cast<int>((idx / w) % h);
  const int nc = static_cast<int>(idx / (static_cast<size_t>(w) * h));
  float a, b;
  match_coeffs(hr_sums, lr_sums, nc, cnt_hr, cnt_lr, &a, &b);
  const float* hp = hb + static_cast<size_t>(nc) * h * w;
  const float* lp = lb + static_cast<size_t>(nc) * h * w;
  const int r = ksize / 2;
  float acc = 0.f;
  for (int dy = 0; dy < ksize; ++dy) {
    const int yy = reflect(y + dy - r, h);
    for (int dx = 0; dx < ksize; ++dx) {
      const int xx = reflect(x + dx - r, w);
      acc += kern[dy * ksize + dx] * (a * hp[yy * w + xx] + b - lp[yy * w + xx]);
    }
  }
  diff[idx] = acc;
}

// 32 consecutive RGB pixels of one warp -> 96 contiguous bytes: 24 word stores assembled with shuffles instead of
// three strided byte stores per thread.  px = b0 | b1 << 8 | b2 << 16; dst = address of lane 0's pixel (4-byte
// aligned); every lane of the warp must call this.
__device__ __forceinline__ void store_rgb_row32(uint8_t* dst, uint32_t px) {
  const int lane = threadIdx.x & 31;
  const int p0 = (4 * lane) / 3, sh = 4 * lane - 3 * p0;  // word `lane` starts `sh` bytes into pixel p0
  const uint32_t lo = __shfl_sync(0xffffffffu, px, p0 & 31), hi = __shfl_sync(0xffffffffu, px, (p0 + 1) & 31);
  const uint64_t two = static_cast<uint64_t>(lo) | (static_cast<uint64_t>(hi) << 24);
  if (lane < 24) reinterpret_cast<uint32_t*>(dst)[lane] = static_cast<uint32_t>(two >> (8 * sh));
}

// ---- finalise: clamp(a*hr + b - bilinear_up(diff), 0, 1) -> uint8 NHWC (truncating) or float NCHW ----------
__global__ void finalize_kernel(Img hr, const float* __restrict__ diff, int dh, int dw, const double* hr_sums,
                                const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* __restrict__ out_u8,
                                float* __restrict__ out_f32, int round_u8) {
  const size_t total = static_cast<size_t>(hr.N) * hr.H * hr.W;
  const size_t idx0 = static_cast<size_t>(blockIdx.x) * blockDim.x;
  const size_t idx = idx0 + threadIdx.x;
  // the match coefficients (double precision, with square roots) once per block and image, not per pixel: a block
  // of 256 consecutive pixels touches at most two images
  __shared__ float coef[2][4][2];
  const size_t plane = static_cast<size_t>(hr.W) * hr.H;
  const int n_first = static_cast<int>(idx0 / plane);
  const bool shared_coef = hr.C <= 4 && plane >= blockDim.x;
  if (threadIdx.x < 2 * hr.C && shared_coef) {
    const int k = threadIdx.x / hr.C, c = threadIdx.x - k * hr.C;
    if (n_first + k < hr.N) match_coeffs(hr_sums, lr_sums, (n_first + k) * hr.C + c, cnt_hr, cnt_lr, &coef[k][c][0], &coef[k][c][1]);
  }
  __syncthreads();
  const bool live = idx < total;
  const size_t idc = live ? idx : total - 1;
  const int x = static_cast<int>(idc % hr.W);
  const int y = static_cast<int>((idc / hr.W) % hr.H);
  const int n = static_cast<int>(idc / plane);
  // bilinear, align_corners=False (area_pixel_compute_source_index): src = (dst + 0.5) * in/out - 0.5, clamped at 0
  int y0 = 0, y1 = 0, x0 = 0, x1 = 0;
  float ly = 0.f, lx = 0.f;
  if (diff != nullptr) {
    float sy = (y + 0.5f) * (static_cast<float>(dh) / hr.H) - 0.5f;
    float sx = (x + 0.5f) * (static_cast<float>(dw) / hr.W) - 0.5f;
    sy = sy < 0.f ? 0.f : sy;
    sx = sx < 0.f ? 0.f : sx;
    y0 = static_cast<int>(sy); x0 = static_cast<int>(sx);
    y1 = y0 < dh - 1 ? y0 + 1 : y0;
    x1 = x0 < dw - 1 ? x0 + 1 : x0;
    ly = sy - y0; lx = sx - x0;
  }
  // whole warp inside the image list and 3 channels: the uint8 row goes out as packed words
  const bool packed = out_u8 != nullptr && hr.C == 3 && __all_sync(0xffffffffu, live) && reinterpret_cast<uintptr_t>(out_u8) % 4 == 0;
  uint32_t px = 0;
  for (int c = 0; c < hr.C; ++c) {
    const int nc = n * hr.C + c;
    float a, b;
    if (shared_coef) { a = coef[n - n_first][c][0]; b = coef[n - n_first][c][1]; }
    else match_coeffs(hr_sums, lr_sums, nc, cnt_hr, cnt_lr, &a, &b);
    float v = a * hr.at(n, c, y, x) + b;
    if (diff != nullptr) {
      const float* d = diff + static_cast<size_t>(nc) * dh * dw;
      const float top = d[y0 * dw + x0] * (1.f - lx) + d[y0 * dw + x1] * lx;
      const float bot = d[y1 * dw + x0] * (1.f - lx) + d[y1 * dw + x1] * lx;
      v -= top * (1.f - ly) + bot * ly;
    }
    v = fminf(fmaxf(v, 0.f), 1.f);
    if (out_u8 != nullptr) {
      float f = v * 255.f;
      if (round_u8) f = rintf(f);
      if (packed) px |= static_cast<uint32_t>(static_cast<uint8_t>(f)) << (8 * c);
      else if (live) out_u8[idx * hr.C + c] = static_cast<uint8_t>(f);
    } else if (live) {
      out_f32[((static_cast<size_t>(n) * hr.C + c) * hr.H + y) * hr.W + x] = v;
    }
  }
  if (packed) store_rgb_row32(out_u8 + (idx - (threadIdx.x & 31)) * 3, px);
}

// ---- bicubic resize (A = -0.75, align_corners=False, clamped taps) of a float NCHW image -> clamp -> uint8 NHWC ----
__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
__global__ void bicubic_u8_kernel(const float* __restrict__ in, int N, int C, int H, int W, uint8_t* __restrict__ out,
                                  int OH, int OW, int round_u8) {
  const size_t total = static_cast<size_t>(N) * OH * OW;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int x = static_cast<int>(idx % OW);
  const int y = static_cast<int>((idx / OW) % OH);
  const int n = static_cast<int>(idx / (static_cast<size_t>(OW) * OH));
  const float A = -0.75f;
  const float sy = (y + 0.5f) * (static_cast<float>(H) / OH) - 0.5f;
  const float sx = (x + 0.5f) * (static_cast<float>(W) / OW) - 0.5f;
  const int iy = static_cast<int>(floorf(sy)), ix = static_cast<int>(floorf(sx));
  const float ty = sy - iy, tx = sx - ix;
  const float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
  const float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
  for (int c = 0; c < C; ++c) {
    const float* p = in + (static_cast<size_t>(n) * C + c) * H * W;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int yy = min(max(iy - 1 + j, 0), H - 1);
      float row = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int xx = min(max(ix - 1 + i, 0), W - 1);
        row += wx[i] * p[static_cast<size_t>(yy) * W + xx];
      }
      acc += wy[j] * row;
    }
    float f = fminf(fmaxf(acc, 0.f), 1.f) * 255.f;
    if (round_u8) f = rintf(f);
    out[idx * C + c] = static_cast<uint8_t>(f);
  }
}

// ---- finalise + bicubic resize in ONE pass: every bicubic tap is clamp(a*hr + b - bilinear_up(diff), 0, 1), so the
//      full-resolution fp32 intermediate of the two-kernel form (708 MB written + read per 4-frame batch at 2880p)
//      never exists.  A block owns a 32 x 8 tile of OUTPUT pixels: it finalises the source patch its taps touch once
//      into shared memory (about 5 evaluations per output pixel at a 2x downscale), then every thread runs its 4x4
//      bicubic from there.  Same arithmetic as finalize_kernel followed by bicubic_u8_kernel
//      (fsrcnn_upscaler.py:214-233).  Source patch limit kFbMaxH x kFbMaxW (downscale factors up to 2).
constexpr int kFbTw = 32, kFbTh = 8, kFbMaxW = 72, kFbMaxH = 24, kFbDiffRows = 6;
// The tile's source patch, finalised into shared memory (both fused kernels): rows py0 .. and columns px0 .. of the
// border-replicated image.  Every thread of the block calls this; it ends with a block-wide barrier.
__device__ __forceinline__ void fb_stage_patch(const Img& hr, const float* __restrict__ diff, int dh, int dw, const double* hr_sums,
                                               const double* lr_sums, double cnt_hr, double cnt_lr, int n, int OH, int OW,
                                               int ox0, int oy0, float fy, float fx, int& py0_out, int& px0_out,
                                               float (&patch)[3][kFbMaxH][kFbMaxW], float (&coef)[3][2],
                                               float (&dxs)[3][kFbDiffRows][kFbMaxW], int (&col_x)[kFbMaxW]) {
  const int H = hr.H, W = hr.W;
  // source patch: rows / columns touched by the taps of the tile's first and last output pixel (before clamping)
  const int oy1 = min(oy0 + kFbTh, OH) - 1, ox1 = min(ox0 + kFbTw, OW) - 1;
  const int py0 = static_cast<int>(floorf((oy0 + 0.5f) * fy - 0.5f)) - 1;
  const int py1 = static_cast<int>(floorf((oy1 + 0.5f) * fy - 0.5f)) + 2;
  const int px0 = static_cast<int>(floorf((ox0 + 0.5f) * fx - 0.5f)) - 1;
  const int px1 = static_cast<int>(floorf((ox1 + 0.5f) * fx - 0.5f)) + 2;
  py0_out = py0;
  px0_out = px0;
  const int ph = py1 - py0 + 1, pw = px1 - px0 + 1;  // host guarantees ph <= kFbMaxH, pw <= kFbMaxW
  // match coefficients (coef): double precision with square roots, once per block
  if (threadIdx.x < 3) match_coeffs(hr_sums, lr_sums, n * hr.C + threadIdx.x, cnt_hr, cnt_lr, &coef[threadIdx.x][0], &coef[threadIdx.x][1]);
  __syncthreads();
  const float ma[3] = {coef[0][0], coef[1][0], coef[2][0]}, mb[3] = {coef[0][1], coef[1][1], coef[2][1]};
  // The bilinear up-sampling of the low-resolution colour difference is separable: interpolate the few diff rows the
  // patch touches along x once per column (dxs), then every patch element needs two shared-memory reads and one
  // lerp per channel instead of twelve global loads and nine lerps.  Same operations in the same order as
  // finalize_kernel (top / bottom row lerps along x, then the lerp along y), so the results are bit-identical.
  int dy_lo = 0;
  bool staged = diff != nullptr;
  if (diff != nullptr) {
    const float ry_scale = static_cast<float>(dh) / H, rx_scale = static_cast<float>(dw) / W;
    {  // diff rows touched by the patch (rows are monotonic in y)
      float s0 = (min(max(py0, 0), H - 1) + 0.5f) * ry_scale - 0.5f, s1 = (min(max(py1, 0), H - 1) + 0.5f) * ry_scale - 0.5f;
      s0 = s0 < 0.f ? 0.f : s0;
      s1 = s1 < 0.f ? 0.f : s1;
      dy_lo = static_cast<int>(s0);
      const int y0l = static_cast<int>(s1);
      const int dy_hi = y0l < dh - 1 ? y0l + 1 : y0l;
      staged = dy_hi - dy_lo + 1 <= kFbDiffRows;
    }
    if (staged) {
      for (int i = threadIdx.x; i < kFbDiffRows * pw; i += kFbTw * kFbTh) {
        const int r = i / pw, rx = i - r * pw;
        const int x = min(max(px0 + rx, 0), W - 1);
        if (r == 0) col_x[rx] = x;
        float sx = (x + 0.5f) * rx_scale - 0.5f;
        sx = sx < 0.f ? 0.f : sx;
        const int x0 = static_cast<int>(sx);
        const int x1 = x0 < dw - 1 ? x0 + 1 : x0;
        const float lx = sx - x0;
        const int yy = dy_lo + r < dh ? dy_lo + r : dh - 1;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float* d = diff + static_cast<size_t>(n * hr.C + c) * dh * dw + static_cast<size_t>(yy) * dw;
          dxs[c][r][rx] = d[x0] * (1.f - lx) + d[x1] * lx;
        }
      }
      __syncthreads();
    }
  }
  if (diff == nullptr || staged) {
    for (int i = threadIdx.x; i < ph * pw; i += kFbTw * kFbTh) {
      const int ry = i / pw, rx = i - ry * pw;
      const int y = min(max(py0 + ry, 0), H - 1);
      int r0 = 0, r1 = 0, x;
      float ly = 0.f;
      if (diff != nullptr) {
        float sy = (y + 0.5f) * (static_cast<float>(dh) / H) - 0.5f;
        sy = sy < 0.f ? 0.f : sy;
        const int y0 = static_cast<int>(sy);
        const int y1 = y0 < dh - 1 ? y0 + 1 : y0;
        ly = sy - y0;
        r0 = y0 - dy_lo;
        r1 = y1 - dy_lo;
        x = col_x[rx];
      } else {
        x = min(max(px0 + rx, 0), W - 1);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float sub = 0.f;
        if (diff != nullptr) sub = dxs[c][r0][rx] * (1.f - ly) + dxs[c][r1][rx] * ly;
        patch[c][ry][rx] = fminf(fmaxf(ma[c] * hr.at(n, c, y, x) + mb[c] - sub, 0.f), 1.f);
      }
    }
  } else
  for (int i = threadIdx.x; i < ph * pw; i += kFbTw * kFbTh) {
    const int ry = i / pw, rx = i - ry * pw;
    const int y = min(max(py0 + ry, 0), H - 1), x = min(max(px0 + rx, 0), W - 1);  // clamped taps (border replicate)
    float sub[3] = {0.f, 0.f, 0.f};
    if (diff != nullptr) {
      float sy = (y + 0.5f) * (static_cast<float>(dh) / H) - 0.5f;
      float sx = (x + 0.5f) * (static_cast<float>(dw) / W) - 0.5f;
      sy = sy < 0.f ? 0.f : sy;
      sx = sx < 0.f ? 0.f : sx;
      const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
      const int y1 = y0 < dh - 1 ? y0 + 1 : y0, x1 = x0 < dw - 1 ? x0 + 1 : x0;
      const float ly = sy - y0, lx = sx - x0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float* d = diff + static_cast<size_t>(n * hr.C + c) * dh * dw;
        const float top = d[y0 * dw + x0] * (1.f - lx) + d[y0 * dw + x1] * lx;
        const float bot = d[y1 * dw + x0] * (1.f - lx) + d[y1 * dw + x1] * lx;
        sub[c] = top * (1.f - ly) + bot * ly;
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) patch[c][ry][rx] = fminf(fmaxf(ma[c] * hr.at(n, c, y, x) + mb[c] - sub[c], 0.f), 1.f);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kFbTw * kFbTh)
finalize_bicubic_u8_kernel(Img hr, const float* __restrict__ diff, int dh, int dw, const double* hr_sums,
                           const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* __restrict__ out,
                           int OH, int OW, int round_u8) {
  __shared__ float patch[3][kFbMaxH][kFbMaxW];
  __shared__ float coef[3][2];
  __shared__ float dxs[3][kFbDiffRows][kFbMaxW];
  __shared__ int col_x[kFbMaxW];
  const int n = blockIdx.z;
  const int ox0 = blockIdx.x * kFbTw, oy0 = blockIdx.y * kFbTh;
  const float fy = static_cast<float>(hr.H) / OH, fx = static_cast<float>(hr.W) / OW;
  int py0, px0;
  fb_stage_patch(hr, diff, dh, dw, hr_sums, lr_sums, cnt_hr, cnt_lr, n, OH, OW, ox0, oy0, fy, fx, py0, px0, patch, coef, dxs, col_x);
  const int x = ox0 + (threadIdx.x % kFbTw), y = oy0 + (threadIdx.x / kFbTw);
  // a warp is one 32-pixel output row of the tile: packed word stores when the whole row is inside the image
  const bool live = x < OW && y < OH;
  const bool packed = __all_sync(0xffffffffu, live) && (static_cast<size_t>(OW) * 3) % 4 == 0 && reinterpret_cast<uintptr_t>(out) % 4 == 0;
  if (!live && !packed) return;
  const float A = -0.75f;
  const float sy = (y + 0.5f) * fy - 0.5f, sx = (x + 0.5f) * fx - 0.5f;
  const int iy = static_cast<int>(floorf(sy)), ix = static_cast<int>(floorf(sx));
  const float ty = sy - iy, tx = sx - ix;
  const float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
  const float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
  const size_t oidx = (static_cast<size_t>(n) * OH + y) * OW + x;
  uint32_t px = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ry = iy - 1 + j - py0;  // the patch already holds the border-replicated value at out-of-image taps
      float row = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) row += wx[i] * patch[c][ry][ix - 1 + i - px0];
      acc += wy[j] * row;
    }
    float f = fminf(fmaxf(acc, 0.f), 1.f) * 255.f;
    if (round_u8) f = rintf(f);
    if (packed) px |= static_cast<uint32_t>(static_cast<uint8_t>(f)) << (8 * c);
    else out[oidx * 3 + c] = static_cast<uint8_t>(f);
  }
  if (packed) store_rgb_row32(out + (oidx - (threadIdx.x & 31)) * 3, px);
}

// ---- NV12 output of the finalising kernels: the uint8 RGB bytes of the kernels above, converted with
//      rgb_to_nv12_kernel's integer arithmetic (elementwise.cu: BT.709 limited range, 15-bit fixed point, chroma = mean
//      of the 2x2 block) and stored as packed frames [N, OH*3/2, OW]: Y plane, then interleaved UV.
// A block of kFbTw x kFbTh threads is a 32 x 8 tile of output pixels whose warp w is row oy0 + w (oy0 % 8 == 0), so the
// two rows of a chroma pair are warps 2k and 2k+1.  Each warp stores its own Y row as packed words; the even warp leaves
// its horizontal pair sums in `xchg`, and after one block-wide barrier the odd warp adds its own and stores the UV row.
// Every thread of the block calls this, dead ones included (rgb then ignored).  OH % 2 == 0 and OW % 4 == 0: a row pair
// is entirely inside or outside the image, and so is each group of 4 lanes.  frame: 4-byte aligned.
__device__ __forceinline__ void store_nv12_tile(uint8_t* frame, int OH, int OW, int x, int y, bool live, const int rgb[3],
                                                uint32_t (&xchg)[kFbTh / 2][kFbTw / 2]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t yv = static_cast<uint32_t>(16 + ((5983 * rgb[0] + 20127 * rgb[1] + 2032 * rgb[2] + 16384) >> 15));
  uint32_t yw = yv | (__shfl_down_sync(0xffffffffu, yv, 1) << 8);
  yw |= __shfl_down_sync(0xffffffffu, yw, 2) << 16;   // lane 4i: Y of pixels 4i .. 4i+3
  const bool st_word = live && (lane & 3) == 0;
  if (st_word) *reinterpret_cast<uint32_t*>(frame + static_cast<size_t>(y) * OW + x) = yw;
  // R, G, B of the pixel pair (lanes 2i, 2i+1) as 10-bit fields: a 2x2 sum is at most 1020
  const uint32_t hs1 = static_cast<uint32_t>(rgb[0]) | (static_cast<uint32_t>(rgb[1]) << 10) | (static_cast<uint32_t>(rgb[2]) << 20);
  const uint32_t hs = hs1 + __shfl_xor_sync(0xffffffffu, hs1, 1);
  uint32_t& slot = xchg[warp >> 1][lane >> 1];
  if ((warp & 1) == 0 && (lane & 1) == 0) slot = hs;
  __syncthreads();
  if (warp & 1) {
    const uint32_t s4 = hs + ((lane & 1) == 0 ? slot : 0u);   // lane 2i: the 2x2 block's sums
    const int sr = static_cast<int>(s4 & 0x3FFu), sg = static_cast<int>((s4 >> 10) & 0x3FFu), sb = static_cast<int>(s4 >> 20);
    const int uu = 128 + ((-3298 * sr - 11094 * sg + 14392 * sb + 65536) >> 17);
    const int vv = 128 + ((14392 * sr - 13073 * sg - 1319 * sb + 65536) >> 17);
    uint32_t uvw = (static_cast<uint32_t>(uu) & 0xFFu) | ((static_cast<uint32_t>(vv) & 0xFFu) << 8);
    uvw |= __shfl_down_sync(0xffffffffu, uvw, 2) << 16;   // lane 4i: U, V of pairs 2i, 2i+1
    if (st_word) *reinterpret_cast<uint32_t*>(frame + static_cast<size_t>(OH) * OW + static_cast<size_t>(y >> 1) * OW + x) = uvw;
  }
}

// finalize_bicubic_u8_kernel with the NV12 store: same tile, patch staging and bicubic taps (same expressions in the
// same order, so the same bytes before the conversion).  No early return: every thread reaches store_nv12_tile's barrier.
__global__ void __launch_bounds__(kFbTw * kFbTh)
finalize_bicubic_nv12_kernel(Img hr, const float* __restrict__ diff, int dh, int dw, const double* hr_sums,
                             const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* __restrict__ out,
                             int OH, int OW, int round_u8) {
  __shared__ float patch[3][kFbMaxH][kFbMaxW];
  __shared__ float coef[3][2];
  __shared__ float dxs[3][kFbDiffRows][kFbMaxW];
  __shared__ int col_x[kFbMaxW];
  __shared__ uint32_t xchg[kFbTh / 2][kFbTw / 2];
  const int n = blockIdx.z;
  const int ox0 = blockIdx.x * kFbTw, oy0 = blockIdx.y * kFbTh;
  const float fy = static_cast<float>(hr.H) / OH, fx = static_cast<float>(hr.W) / OW;
  int py0, px0;
  fb_stage_patch(hr, diff, dh, dw, hr_sums, lr_sums, cnt_hr, cnt_lr, n, OH, OW, ox0, oy0, fy, fx, py0, px0, patch, coef, dxs, col_x);
  const int x = ox0 + (threadIdx.x % kFbTw), y = oy0 + (threadIdx.x / kFbTw);
  const bool live = x < OW && y < OH;
  int rgb[3] = {0, 0, 0};
  if (live) {
    const float A = -0.75f;
    const float sy = (y + 0.5f) * fy - 0.5f, sx = (x + 0.5f) * fx - 0.5f;
    const int iy = static_cast<int>(floorf(sy)), ix = static_cast<int>(floorf(sx));
    const float ty = sy - iy, tx = sx - ix;
    const float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
    const float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int ry = iy - 1 + j - py0;
        float row = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) row += wx[i] * patch[c][ry][ix - 1 + i - px0];
        acc += wy[j] * row;
      }
      float f = fminf(fmaxf(acc, 0.f), 1.f) * 255.f;
      if (round_u8) f = rintf(f);
      rgb[c] = static_cast<uint8_t>(f);
    }
  }
  store_nv12_tile(out + static_cast<size_t>(n) * OH * OW * 3 / 2, OH, OW, x, y, live, rgb, xchg);
}

// finalize_kernel's uint8 arithmetic (match affine, bilinear up-sampling of diff, clamp, x255, truncation or rint; same
// expressions in the same order) on a 2-D grid of 32 x 8 tiles, blockIdx.z = image, with the NV12 store.  C == 3.
__global__ void __launch_bounds__(kFbTw * kFbTh)
finalize_nv12_kernel(Img hr, const float* __restrict__ diff, int dh, int dw, const double* hr_sums, const double* lr_sums,
                     double cnt_hr, double cnt_lr, uint8_t* __restrict__ out, int round_u8) {
  __shared__ float coef[3][2];
  __shared__ uint32_t xchg[kFbTh / 2][kFbTw / 2];
  const int n = blockIdx.z;
  if (threadIdx.x < 3) match_coeffs(hr_sums, lr_sums, n * 3 + threadIdx.x, cnt_hr, cnt_lr, &coef[threadIdx.x][0], &coef[threadIdx.x][1]);
  __syncthreads();
  const int x = blockIdx.x * kFbTw + (threadIdx.x % kFbTw), y = blockIdx.y * kFbTh + (threadIdx.x / kFbTw);
  const bool live = x < hr.W && y < hr.H;
  int rgb[3] = {0, 0, 0};
  if (live) {
    int y0 = 0, y1 = 0, x0 = 0, x1 = 0;
    float ly = 0.f, lx = 0.f;
    if (diff != nullptr) {
      float sy = (y + 0.5f) * (static_cast<float>(dh) / hr.H) - 0.5f;
      float sx = (x + 0.5f) * (static_cast<float>(dw) / hr.W) - 0.5f;
      sy = sy < 0.f ? 0.f : sy;
      sx = sx < 0.f ? 0.f : sx;
      y0 = static_cast<int>(sy); x0 = static_cast<int>(sx);
      y1 = y0 < dh - 1 ? y0 + 1 : y0;
      x1 = x0 < dw - 1 ? x0 + 1 : x0;
      ly = sy - y0; lx = sx - x0;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v = coef[c][0] * hr.at(n, c, y, x) + coef[c][1];
      if (diff != nullptr) {
        const float* d = diff + static_cast<size_t>(n * 3 + c) * dh * dw;
        const float top = d[y0 * dw + x0] * (1.f - lx) + d[y0 * dw + x1] * lx;
        const float bot = d[y1 * dw + x0] * (1.f - lx) + d[y1 * dw + x1] * lx;
        v -= top * (1.f - ly) + bot * ly;
      }
      v = fminf(fmaxf(v, 0.f), 1.f);
      float f = v * 255.f;
      if (round_u8) f = rintf(f);
      rgb[c] = static_cast<uint8_t>(f);
    }
  }
  store_nv12_tile(out + static_cast<size_t>(n) * hr.H * hr.W * 3 / 2, hr.H, hr.W, x, y, live, rgb, xchg);
}

// ---- 3x3 depthwise reflect "sharpen" + clamp, optional blend with another image (float NCHW in/out) ----------
//   out = opacity * clamp(sum k[dy][dx] * x[reflect], 0, 1) + (1 - opacity) * other
__global__ void sharpen_blend_kernel(Img x, float k_center, float k_side, float opacity, Img other, float* __restrict__ out) {
  const size_t total = static_cast<size_t>(x.N) * x.C * x.H * x.W;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int px = static_cast<int>(idx % x.W);
  const int py = static_cast<int>((idx / x.W) % x.H);
  const int c = static_cast<int>((idx / (static_cast<size_t>(x.W) * x.H)) % x.C);
  const int n = static_cast<int>(idx / (static_cast<size_t>(x.W) * x.H * x.C));
  float acc = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
      acc += ((dy == 0 && dx == 0) ? k_center : k_side) * x.at(n, c, reflect(py + dy, x.H), reflect(px + dx, x.W));
  float v = fminf(fmaxf(acc, 0.f), 1.f);
  if (other.p != nullptr) v = opacity * v + (1.f - opacity) * other.at(n, c, py, px);
  out[idx] = v;
}

// The same arithmetic, written as the upscaler's first-layer activation tensor: 16-bit NHWC [N, H/us, W/us, pitch] with
// torch pixel_unshuffle(us) channel order (ch = c*us*us + iy*us + jx), zero channel padding -- what the plan's layout
// kernel would produce from the float image (prep_kernel, elementwise.cu), without the float image.
__global__ void sharpen_blend_act_kernel(Img x, float k_center, float k_side, float opacity, Img other, uint16_t* __restrict__ out,
                                         int us, int pitch, int bf16) {
  const int OH = x.H / us, OW = x.W / us;
  const size_t total = static_cast<size_t>(x.N) * OH * OW;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ox = static_cast<int>(idx % OW);
  const int oy = static_cast<int>((idx / OW) % OH);
  const int n = static_cast<int>(idx / (static_cast<size_t>(OW) * OH));
  const int creal = x.C * us * us;
  uint16_t* o = out + idx * pitch;
  for (int c8 = 0; c8 < pitch; c8 += 8) {
    uint16_t v8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int ch = c8 + i;
      float v = 0.f;
      if (ch < creal) {
        const int c = ch / (us * us), rem = ch - c * us * us;
        const int py = oy * us + rem / us, px = ox * us + rem % us;
        float acc = 0.f;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx)
            acc += ((dy == 0 && dx == 0) ? k_center : k_side) * x.at(n, c, reflect(py + dy, x.H), reflect(px + dx, x.W));
        v = fminf(fmaxf(acc, 0.f), 1.f);
        if (other.p != nullptr) v = opacity * v + (1.f - opacity) * other.at(n, c, py, px);
      }
      if (bf16) { const __nv_bfloat16 h = __float2bfloat16_rn(v); v8[i] = *reinterpret_cast<const uint16_t*>(&h); }
      else { const __half h = __float2half_rn(v); v8[i] = *reinterpret_cast<const uint16_t*>(&h); }
    }
    *reinterpret_cast<uint4*>(o + c8) = *reinterpret_cast<const uint4*>(v8);
  }
}

// Hot case of the cfg3 hand-over (RRDBNet x2: pixel_unshuffle(2), 3 channels, denoised frame as half NCHW, original
// frame as NV12 or uint8 RGB): one thread per trunk pixel = a 2x2 block of the frame.  It loads the 4x4 patch of each
// channel once (48 values instead of 108 gathers) and the block's four luma / one chroma sample(s); the arithmetic and
// its order are those of sharpen_blend_act_kernel (same expressions -> bit-identical results, tests/test_cfg3_gpu.py).
__global__ void sharpen_blend_act_us2_kernel(const __half* __restrict__ x, int N, int H, int W, float k_center, float k_side,
                                             float opacity, const uint8_t* __restrict__ other, int other_fmt,
                                             uint16_t* __restrict__ out, int pitch) {
  const int OH = H >> 1, OW = W >> 1;
  const size_t total = static_cast<size_t>(N) * OH * OW;
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ox = static_cast<int>(idx % OW);
  const int oy = static_cast<int>((idx / OW) % OH);
  const int n = static_cast<int>(idx / (static_cast<size_t>(OW) * OH));
  int ry[4], rx[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    ry[i] = reflect(2 * oy - 1 + i, H);
    rx[i] = reflect(2 * ox - 1 + i, W);
  }
  // the original frame's 2x2 block: [iy][jx][c]
  float org[2][2][3];
  if (other != nullptr) {
    if (other_fmt == 3) {
      const uint8_t* frame = other + static_cast<size_t>(n) * (static_cast<size_t>(H) * W * 3 / 2);
      const uint8_t* uv = frame + static_cast<size_t>(H) * W + static_cast<size_t>(oy) * W + 2 * ox;
      const float cb = (static_cast<float>(uv[0]) - 128.f) * (1.f / 224.f), cr = (static_cast<float>(uv[1]) - 128.f) * (1.f / 224.f);
#pragma unroll
      for (int iy = 0; iy < 2; ++iy)
#pragma unroll
        for (int jx = 0; jx < 2; ++jx) {
          const float yy = (static_cast<float>(frame[static_cast<size_t>(2 * oy + iy) * W + 2 * ox + jx]) - 16.f) * (1.f / 219.f);
          org[iy][jx][0] = fminf(fmaxf(yy + 1.5748f * cr, 0.f), 1.f);
          org[iy][jx][1] = fminf(fmaxf(yy - 0.187324f * cb - 0.468124f * cr, 0.f), 1.f);
          org[iy][jx][2] = fminf(fmaxf(yy + 1.8556f * cb, 0.f), 1.f);
        }
    } else {
#pragma unroll
      for (int iy = 0; iy < 2; ++iy)
#pragma unroll
        for (int jx = 0; jx < 2; ++jx)
#pragma unroll
          for (int c = 0; c < 3; ++c)
            org[iy][jx][c] = static_cast<float>(other[((static_cast<size_t>(n) * H + 2 * oy + iy) * W + 2 * ox + jx) * 3 + c]) / 255.0f;
    }
  }
  uint16_t v16[16];
#pragma unroll
  for (int i = 12; i < 16; ++i) v16[i] = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const __half* plane = x + (static_cast<size_t>(n) * 3 + c) * H * W;
    float p[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) p[i][j] = __half2float(plane[static_cast<size_t>(ry[i]) * W + rx[j]]);
#pragma unroll
    for (int iy = 0; iy < 2; ++iy)
#pragma unroll
      for (int jx = 0; jx < 2; ++jx) {
        float acc = 0.f;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx)
            acc += ((dy == 0 && dx == 0) ? k_center : k_side) * p[iy + dy + 1][jx + dx + 1];
        float v = fminf(fmaxf(acc, 0.f), 1.f);
        if (other != nullptr) v = opacity * v + (1.f - opacity) * org[iy][jx][c];
        const __half h = __float2half_rn(v);
        v16[c * 4 + iy * 2 + jx] = *reinterpret_cast<const uint16_t*>(&h);
      }
  }
  uint16_t* o = out + idx * pitch;
  *reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(v16);
  *reinterpret_cast<uint4*>(o + 8) = *reinterpret_cast<const uint4*>(v16 + 8);
  for (int c8 = 16; c8 < pitch; c8 += 8) *reinterpret_cast<uint4*>(o + c8) = make_uint4(0u, 0u, 0u, 0u);
}

inline unsigned blocks_for(size_t total, int threads) { return static_cast<unsigned>((total + threads - 1) / threads); }

}  // namespace
}  // namespace ss4k

using namespace ss4k;

extern "C" {

int ss4k_glue_chan_stats(const void* img, int fmt, int n, int c, int h, int w, double* sums_dev, void* stream) {
  if (!img || !sums_dev || fmt < 0 || fmt > 2) return SS4K_E_INVALID;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(sums_dev, 0, sizeof(double) * 2 * n * c, st) != cudaSuccess) return SS4K_E_CUDA;
  const size_t total = static_cast<size_t>(h) * w;
  if (fmt == 1 && total % 8 == 0 && reinterpret_cast<uintptr_t>(img) % 16 == 0) {
    const size_t vec = total / 8;
    const unsigned gx = static_cast<unsigned>(std::min<size_t>((vec + 255) / 256, std::max(1, 1184 / (n * c))));  // ~8 blocks per SM in all
    chan_stats_half_kernel<<<dim3(gx, static_cast<unsigned>(n * c)), 256, 0, st>>>(reinterpret_cast<const uint4*>(img), vec, sums_dev);
    return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
  }
  dim3 grid(static_cast<unsigned>(std::min<size_t>((total + 1023) / 1024, 296)), static_cast<unsigned>(n * c));
  chan_stats_kernel<<<grid, 256, 0, st>>>(Img{img, fmt, n, c, h, w}, sums_dev);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_area_pool(const void* img, int fmt, int n, int c, int h, int w, float* out_dev, int oh, int ow, void* stream) {
  if (!img || !out_dev || fmt < 0 || fmt > 2 || n < 1 || c < 1 || h < 1 || w < 1 || oh < 1 || ow < 1) return SS4K_E_INVALID;
  const size_t total = static_cast<size_t>(n) * c * oh * ow;
  area_pool_kernel<<<blocks_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(Img{img, fmt, n, c, h, w}, out_dev, oh, ow);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_blur_diff(const float* hb, const float* lb, float* diff, const float* kern_dev, int ksize, int n, int c, int h,
                        int w, const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, void* stream) {
  if (!hb || !lb || !diff || !kern_dev || n < 1 || c < 1) return SS4K_E_INVALID;
  // reflect() mirrors an index once: the radius must stay below both sizes (F.pad(mode='reflect') refuses the rest)
  if (ksize < 1 || ksize % 2 == 0 || ksize / 2 >= h || ksize / 2 >= w) return SS4K_E_INVALID;
  const size_t total = static_cast<size_t>(n) * c * h * w;
  blur_diff_kernel<<<blocks_for(total, 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(hb, lb, diff, kern_dev, ksize, n, c, h, w,
                                                                                           hr_sums, lr_sums, cnt_hr, cnt_lr);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_finalize(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                       const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* out_u8,
                       float* out_f32, int round_u8, void* stream) {
  if (!hr || (!out_u8 && !out_f32) || fmt < 0 || fmt > 1) return SS4K_E_INVALID;
  if (diff && (dh < 1 || dw < 1)) return SS4K_E_INVALID;
  const size_t total = static_cast<size_t>(n) * h * w;
  finalize_kernel<<<blocks_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(Img{hr, fmt, n, c, h, w}, diff, dh, dw, hr_sums,
                                                                                          lr_sums, cnt_hr, cnt_lr, out_u8, out_f32, round_u8);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_finalize_bicubic_u8(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                                  const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* out_u8,
                                  int oh, int ow, int round_u8, void* stream) {
  if (!hr || !out_u8 || fmt < 0 || fmt > 1 || c != 3 || oh <= 0 || ow <= 0) return SS4K_E_INVALID;
  if (diff && (dh < 1 || dw < 1)) return SS4K_E_INVALID;
  // the tile kernel's shared-memory patch covers downscale factors up to 2 (plus the 3-pixel tap margin)
  const double fy = static_cast<double>(h) / oh, fx = static_cast<double>(w) / ow;
  if (fy * (kFbTh - 1) + 5.0 > kFbMaxH || fx * (kFbTw - 1) + 5.0 > kFbMaxW) return SS4K_E_INVALID;
  dim3 grid((ow + kFbTw - 1) / kFbTw, (oh + kFbTh - 1) / kFbTh, n);
  finalize_bicubic_u8_kernel<<<grid, kFbTw * kFbTh, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      Img{hr, fmt, n, c, h, w}, diff, dh, dw, hr_sums, lr_sums, cnt_hr, cnt_lr, out_u8, oh, ow, round_u8);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_finalize_nv12(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                            const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* out_nv12,
                            int round_u8, void* stream) {
  if (!hr || !out_nv12 || fmt < 0 || fmt > 1 || c != 3 || n < 1 || h < 1 || w < 1) return SS4K_E_INVALID;
  if (h % 2 || w % 4 || reinterpret_cast<uintptr_t>(out_nv12) % 4) return SS4K_E_INVALID;
  if (diff && (dh < 1 || dw < 1)) return SS4K_E_INVALID;
  dim3 grid((w + kFbTw - 1) / kFbTw, (h + kFbTh - 1) / kFbTh, n);
  finalize_nv12_kernel<<<grid, kFbTw * kFbTh, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      Img{hr, fmt, n, c, h, w}, diff, dh, dw, hr_sums, lr_sums, cnt_hr, cnt_lr, out_nv12, round_u8);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_finalize_bicubic_nv12(const void* hr, int fmt, int n, int c, int h, int w, const float* diff, int dh, int dw,
                                    const double* hr_sums, const double* lr_sums, double cnt_hr, double cnt_lr, uint8_t* out_nv12,
                                    int oh, int ow, int round_u8, void* stream) {
  if (!hr || !out_nv12 || fmt < 0 || fmt > 1 || c != 3 || oh <= 0 || ow <= 0) return SS4K_E_INVALID;
  if (oh % 2 || ow % 4 || reinterpret_cast<uintptr_t>(out_nv12) % 4) return SS4K_E_INVALID;
  if (diff && (dh < 1 || dw < 1)) return SS4K_E_INVALID;
  const double fy = static_cast<double>(h) / oh, fx = static_cast<double>(w) / ow;   // same patch guard as the uint8 entry
  if (fy * (kFbTh - 1) + 5.0 > kFbMaxH || fx * (kFbTw - 1) + 5.0 > kFbMaxW) return SS4K_E_INVALID;
  dim3 grid((ow + kFbTw - 1) / kFbTw, (oh + kFbTh - 1) / kFbTh, n);
  finalize_bicubic_nv12_kernel<<<grid, kFbTw * kFbTh, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      Img{hr, fmt, n, c, h, w}, diff, dh, dw, hr_sums, lr_sums, cnt_hr, cnt_lr, out_nv12, oh, ow, round_u8);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_bicubic_u8(const float* in, int n, int c, int h, int w, uint8_t* out, int oh, int ow, int round_u8, void* stream) {
  if (!in || !out || n < 1 || c < 1 || h < 1 || w < 1 || oh < 1 || ow < 1) return SS4K_E_INVALID;
  const size_t total = static_cast<size_t>(n) * oh * ow;
  bicubic_u8_kernel<<<blocks_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(in, n, c, h, w, out, oh, ow, round_u8);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

int ss4k_glue_sharpen_blend(const void* x, int fmt, int n, int c, int h, int w, float strength, float opacity, const void* other,
                            int other_fmt, float* out, void* stream) {
  if (!x || !out || fmt < 0 || fmt > 2 || (other && (other_fmt < 0 || other_fmt > 3))) return SS4K_E_INVALID;
  if (h < 2 || w < 2) return SS4K_E_INVALID;  // the 3x3 reflect needs a neighbour on each side
  // sharpen_ker (fsrcnn_upscaler.py:54-84): (sharp*s + identity*(1-s)) / sum, sharp = [-1..9..-1]
  const float center = 9.f * strength + (1.f - strength), side = -strength;
  const float sum = center + 8.f * side;
  const size_t total = static_cast<size_t>(n) * c * h * w;
  sharpen_blend_kernel<<<blocks_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      Img{x, fmt, n, c, h, w}, center / sum, side / sum, opacity, Img{other, other_fmt, n, c, h, w}, out);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

// ss4k_glue_sharpen_blend with the result written as a plan's first-layer activation tensor (ss4k_plan_input_act): the glue
// between the denoiser and the upscaler (fsrcnn_upscaler.py:278-281) then feeds conv_first directly -- no float image, no
// layout kernel in the upscaler's plan (ss4k_run_act).
int ss4k_glue_sharpen_blend_act(const void* x, int fmt, int n, int c, int h, int w, float strength, float opacity, const void* other,
                                int other_fmt, void* act_out, int unshuffle, int pitch, int bf16, void* stream) {
  if (!x || !act_out || fmt < 0 || fmt > 2 || (other && (other_fmt < 0 || other_fmt > 3))) return SS4K_E_INVALID;
  if (h < 2 || w < 2) return SS4K_E_INVALID;
  if (unshuffle < 1 || h % unshuffle || w % unshuffle || pitch % 8 || pitch < c * unshuffle * unshuffle) return SS4K_E_INVALID;
  const float center = 9.f * strength + (1.f - strength), side = -strength;
  const float sum = center + 8.f * side;
  const size_t total = static_cast<size_t>(n) * (h / unshuffle) * (w / unshuffle);
  if (unshuffle == 2 && c == 3 && fmt == 1 && !bf16 && pitch >= 16 && (!other || other_fmt == 2 || other_fmt == 3) &&
      getenv("SS4K_GLUE_GENERIC") == nullptr) {
    sharpen_blend_act_us2_kernel<<<blocks_for(total, 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const __half*>(x), n, h, w, center / sum, side / sum, opacity, reinterpret_cast<const uint8_t*>(other), other_fmt,
        reinterpret_cast<uint16_t*>(act_out), pitch);
    return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
  }
  sharpen_blend_act_kernel<<<blocks_for(total, 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      Img{x, fmt, n, c, h, w}, center / sum, side / sum, opacity, Img{other, other_fmt, n, c, h, w},
      reinterpret_cast<uint16_t*>(act_out), unshuffle, pitch, bf16);
  return cudaGetLastError() == cudaSuccess ? SS4K_OK : SS4K_E_CUDA;
}

}  // extern "C"
