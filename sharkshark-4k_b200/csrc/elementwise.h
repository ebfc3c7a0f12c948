#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv_params.h"

namespace ss4k {

// conv_tc.cu
cudaError_t conv_tc_prepare();
cudaError_t conv_tc_launch(const ConvParams& p, int grid, cudaStream_t stream);

// conv_stream.cu
cudaError_t conv_stream_prepare();
cudaError_t conv_stream_launch(const StreamParams& p, int nout, int grid, cudaStream_t stream, bool pdl);
int conv_stream_max_ctas_per_sm(int nout);  // resident CTAs per SM of the variant (early activation loads need exactly 1)

// tiled inference: one padded crop of the (reflect-padded) frame and where its un-padded centre goes in the output
struct TileBox {
  int32_t src_y, src_x;       // top-left of the padded crop in the input frame
  int32_t off_y, off_x;       // top-left of the un-padded centre inside the net's output for the crop (pixels of the output grid)
  int32_t dst_y, dst_x;       // where it goes in the output frame
  int32_t paste_h, paste_w;   // its size (clipped to the output frame by the kernel)
  int32_t crop_h, crop_w;     // size of the padded crop
  int32_t img, atlas_x;       // atlas image of the group it is packed into and its column there (crops sit side by side,
                              // top-aligned, zero gap columns between them; the rest of the hc x wc canvas is zero)
};
// fmt: SS4K_FMT_F32_NCHW / F16_NCHW / U8_NHWC; the crops are packed into nimg atlas images per frame, stored as a batch
// [img * N + n] of hc x wc images in the same format
cudaError_t tile_gather_launch(int fmt, const void* in, void* out, const TileBox* boxes_dev, int nbox, int nimg, int N, int C, int H,
                               int W, int pre_pad, int hc, int wc, cudaStream_t s);
cudaError_t tile_paste_launch(int fmt, const void* crops, void* out, const TileBox* boxes_dev, int nbox, int N, int C, int hco,
                              int wco, int scale, int OH, int OW, cudaStream_t s);

// elementwise.cu
// in_fmt: SS4K_FMT_* ; out: [N, H/us, W/us, pitch] 16-bit NHWC (out_lo: low halves for split mode or null)
cudaError_t prep_launch(int in_fmt, const void* in, void* out, void* out_lo, int N, int C, int H, int W,
                        int pitch, int unshuffle, int fill_ch, float fill_val, int bf16, cudaStream_t s);
// uint8 NHWC RGB [N,H,W,3] -> NV12 (Y plane + interleaved UV per frame), BT.709 limited range, H % 2 == 0, W % 4 == 0
cudaError_t rgb_to_nv12_launch(const void* rgb, void* nv12, int N, int H, int W, cudaStream_t s);
cudaError_t unprep_launch(const void* in, const void* in_lo, float* out, int N, int C, int H, int W,
                          int pitch, int coff, int bf16, cudaStream_t s);
cudaError_t ref_conv3x3_launch(const void* in, const float* w, const float* bias, float* out, int N, int H,
                               int W, int pitch, int cin, int cout, int bf16, cudaStream_t s);

}  // namespace ss4k
