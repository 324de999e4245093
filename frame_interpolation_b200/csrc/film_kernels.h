// Launchers of the bandwidth-bound (non-GEMM) kernels of the FILM engine.
#pragma once
#include <cuda_runtime.h>

#include "film_common.cuh"

namespace film {

// util.py:38-44 -- 2x2/2 VALID average pool of a 3-channel fp32 image batch.
cudaError_t launch_image_pool(const float* in, float* out, int B, int H, int W, cudaStream_t st);

// feature_extractor.py:119 (cfeat_conv_0: 3 -> 64, 3x3 SAME, LeakyReLU): K = 27, HBM-bound.
// w: [27][64] fp32 (k = (ky*3+kx)*3 + ci), writes split output into a channel slice.
cudaError_t launch_conv0_c3(const float* img, int B, int H, int W, const float* w,
                            const float* bias, sp_t* out_hi, sp_t* out_lo, int out_C,
                            int out_c_off, cudaStream_t st);

// Product path of cfeat_conv_0: register-tiled fp32 direct conv (K = 27 is too short for the tensor cores), reads the
// fp32 image level, writes the 64-channel split output [B][H][W][64] (hi plane only when `lo_skip`).
// `pool_out` (nullable): [B][H/2][W/2][3] fp32 -- the 2x2/2 VALID average pool of `img` (util.py:38-44), i.e. the next
// image pyramid level, written from the input patch the conv has staged anyway (sizes floor: an odd last row / column
// is dropped).
cudaError_t launch_fe_conv0(const float* img, int B, int H, int W, const float* w, const float* bias, sp_t* out_hi,
                            sp_t* out_lo, bool lo_skip, float* pool_out, cudaStream_t st);

// im2col-lite for the tensor-core version of cfeat_conv_0: [B][H][W][3] fp32 -> [B][H][W][32] split
// (27 tap x channel values in HWIO order + 5 zero channels, zero outside the image).
cudaError_t launch_im2col3x3(const float* img, int B, int H, int W, sp_t* out_hi, sp_t* out_lo, cudaStream_t st);

// [B][H][W][3] fp32 -> channels 0..7 of a zero-initialised [B][H][W][32] split tensor (3 real channels).
cudaError_t launch_image_to_split32(const float* img, int B, int H, int W, sp_t* out_hi, sp_t* out_lo, cudaStream_t st);

// feature_extractor.py:138-146 -- 2x2/2 VALID average pool of a channel slice of a split tensor.
cudaError_t launch_act_pool(const sp_t* in_hi, const sp_t* in_lo, int in_C, int in_c_off, int B,
                            int H, int W, int Cn, sp_t* out_hi, sp_t* out_lo, int out_C,
                            cudaStream_t st);

// fusion.py:133 -- nearest-neighbour resize (TF2 rule, fp32 index arithmetic) of a split tensor
// [B][Hc][Wc][C] -> [B][Hf][Wf][C], C a multiple of 8: the decoder's up-sampling at levels where the fine grid is
// not twice the coarse one.  hi_only: only the hi plane is copied (single-pass consumer).
cudaError_t launch_resize_nearest(const sp_t* in_hi, const sp_t* in_lo, int B, int Hc, int Wc, int C, sp_t* out_hi,
                                  sp_t* out_lo, int Hf, int Wf, bool hi_only, cudaStream_t st);

// pyramid_flow_estimator.py:154-157 fused: v_up = resize_bilinear(2*v_prev -> HxW);
// warped[d] = warp(feat[1-d], v_up[d]).  feat/warped are [2][H][W][C] split tensors.
cudaError_t launch_flow_warp(const float* v_prev, int Hc, int Wc, const sp_t* feat_hi,
                             const sp_t* feat_lo, int H, int W, int C, float* v_up,
                             sp_t* warped_hi, sp_t* warped_lo, bool hi_only, cudaStream_t st);
// hi_only (both gathers): the destination's only consumers are single-pass convs -> read and write the hi
// planes alone (half the bytes; the lo planes of the destination are left untouched and never read)

// pyramid_flow_estimator.py:77-83,96-97 (conv_3: 1x1 nf->nf/2 LReLU, conv_4: 1x1 ->2 linear)
// fused with :161 (v = v_residual + v).  x: [2][H][W][Cx] split (first nf channels real).
cudaError_t launch_flow_head(const sp_t* x_hi, const sp_t* x_lo, int Cx, int nf, int npix,
                             const float* w3, const float* b3, const float* w4, const float* b4,
                             const float* v_up, float* residual, float* v, cudaStream_t st);

// interpolator.py:163-183: flows * 0.5, warp of [image, features] pyramids.
// warped[k] = warp(feat[k], 0.5 * v[1-k])   (k = 0: image 0 by backward flow, k = 1: image 1
// by forward flow; v[0] = forward flow, v[1] = backward flow).
cudaError_t launch_fusion_warp(const float* v, const sp_t* feat_hi, const sp_t* feat_lo, int H,
                               int W, int C, sp_t* warped_hi, sp_t* warped_lo, bool hi_only, cudaStream_t st);
// side tensor [1][H][W][side_C] split: ch 0-2 warp(img0, .5*bwd), 3-5 warp(img1, .5*fwd),
// 6-7 .5*bwd, 8-9 .5*fwd, 10-15 zero.
cudaError_t launch_fusion_side(const float* v, const float* img, int H, int W, sp_t* side_hi,
                               sp_t* side_lo, int side_C, cudaStream_t st);

// fusion.py:100-101,139 (1x1 conv 64 -> 3, linear) + crop (eval/interpolator.py:175).
cudaError_t launch_rgb_head(const sp_t* x_hi, const sp_t* x_lo, int Cx, int H, int W,
                            const float* w, const float* b, float* out, int64_t out_pitch,
                            int off_y, int off_x, int out_h, int out_w, cudaStream_t st);

// zero-pad copy (eval/interpolator.py:56): dst [H][W][3] <- src [h][w][3] at (off_y, off_x).
cudaError_t launch_pad_image(const float* src, int64_t src_pitch, int h, int w, float* dst, int H,
                             int W, int off_y, int off_x, cudaStream_t st);

// 8-bit front / back end: eval/util.py:38-41 (uint8 / 255 -> float32) and :51-52 (clip(x * 255, 0, 255) + 0.5 -> uint8)
cudaError_t launch_u8_to_f32(const uint8_t* src, float* dst, int64_t n, cudaStream_t st);
cudaError_t launch_f32_to_u8(const float* src, uint8_t* dst, int64_t n, cudaStream_t st);

// debug: split tensor slice -> fp32 NHWC
cudaError_t launch_unsplit(const sp_t* hi, const sp_t* lo, int C, int c_off, int Cn, int64_t npix,
                           float* out, cudaStream_t st);

}  // namespace film
