// Bandwidth-bound kernels of the FILM engine (sm_100a): pooling, first conv (K = 27),
// flow-upsample + warp gathers, flow / RGB heads, and the CUDA-core validation conv.
// All activations are NHWC; feature tensors are in the split 2 x 16-bit format
// (film_common.cuh).  Every kernel reads/writes 128-bit channel vectors.
#include "film_conv.h"
#include "film_kernels.h"

namespace film {

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// ------------------------------------------------------------------------------------------
// util.py:38-44  image pyramid pool (fp32, 3 channels)
// ------------------------------------------------------------------------------------------
__global__ void k_image_pool(const float* __restrict__ in, float* __restrict__ out, int B, int H,
                             int W) {
  const int Ho = H / 2, Wo = W / 2;
  const int64_t n = (int64_t)B * Ho * Wo * 3;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % 3);
  int64_t p = i / 3;
  int x = (int)(p % Wo);
  p /= Wo;
  int y = (int)(p % Ho);
  int b = (int)(p / Ho);
  const float* r0 = in + (((int64_t)b * H + 2 * y) * W + 2 * x) * 3 + c;
  const float* r1 = r0 + (int64_t)W * 3;
  out[i] = (r0[0] + r0[3] + r1[0] + r1[3]) * 0.25f;
}

cudaError_t launch_image_pool(const float* in, float* out, int B, int H, int W, cudaStream_t st) {
  int64_t n = (int64_t)B * (H / 2) * (W / 2) * 3;
  if (n == 0) return cudaSuccess;
  k_image_pool<<<cdiv(n, 256), 256, 0, st>>>(in, out, B, H, W);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// eval/interpolator.py:56  zero-pad copy
// ------------------------------------------------------------------------------------------
__global__ void k_pad_image(const float* __restrict__ src, int64_t src_pitch, int h, int w,
                            float* __restrict__ dst, int H, int W, int off_y, int off_x) {
  const int64_t n = (int64_t)H * W * 3;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % 3);
  int64_t p = i / 3;
  int x = (int)(p % W), y = (int)(p / W);
  int sy = y - off_y, sx = x - off_x;
  float v = 0.f;
  if (sy >= 0 && sy < h && sx >= 0 && sx < w) v = src[(int64_t)sy * src_pitch + sx * 3 + c];
  dst[i] = v;
}

cudaError_t launch_pad_image(const float* src, int64_t src_pitch, int h, int w, float* dst, int H,
                             int W, int off_y, int off_x, cudaStream_t st) {
  int64_t n = (int64_t)H * W * 3;
  k_pad_image<<<cdiv(n, 256), 256, 0, st>>>(src, src_pitch, h, w, dst, H, W, off_y, off_x);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// 8-bit front / back end (SURVEY 8f row 3).  eval/util.py:38-41: image = uint8 / 255 (float32 division);
// eval/util.py:51-52: uint8 = trunc(clip(image * 255, 0, 255) + 0.5), every step rounded to float32 like numpy.
// ------------------------------------------------------------------------------------------
template <bool kVec>
__global__ void __launch_bounds__(256) k_u8_to_f32(const uint8_t* __restrict__ src, float* __restrict__ dst, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (kVec && i + 3 < n) {
    const uchar4 u = *reinterpret_cast<const uchar4*>(src + i);
    float4 f;
    f.x = __fdiv_rn((float)u.x, 255.f);
    f.y = __fdiv_rn((float)u.y, 255.f);
    f.z = __fdiv_rn((float)u.z, 255.f);
    f.w = __fdiv_rn((float)u.w, 255.f);
    *reinterpret_cast<float4*>(dst + i) = f;
  } else {
    for (int64_t j = i; j < n && j < i + 4; ++j) dst[j] = __fdiv_rn((float)src[j], 255.f);
  }
}
__device__ __forceinline__ uint8_t quantize_u8(float x) {
  const float s = fminf(fmaxf(__fmul_rn(x, 255.f), 0.f), 255.f);
  return (uint8_t)__fadd_rn(s, 0.5f);  // truncation, like numpy's astype(uint8)
}
template <bool kVec>
__global__ void __launch_bounds__(256) k_f32_to_u8(const float* __restrict__ src, uint8_t* __restrict__ dst, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (kVec && i + 3 < n) {
    const float4 f = *reinterpret_cast<const float4*>(src + i);
    uchar4 u;
    u.x = quantize_u8(f.x);
    u.y = quantize_u8(f.y);
    u.z = quantize_u8(f.z);
    u.w = quantize_u8(f.w);
    *reinterpret_cast<uchar4*>(dst + i) = u;
  } else {
    for (int64_t j = i; j < n && j < i + 4; ++j) dst[j] = quantize_u8(src[j]);
  }
}
cudaError_t launch_u8_to_f32(const uint8_t* src, float* dst, int64_t n, cudaStream_t st) {
  // vector accesses need a 4-byte aligned source and a 16-byte aligned destination (frame slots of odd sizes are not)
  const bool vec = ((uintptr_t)src & 3) == 0 && ((uintptr_t)dst & 15) == 0;
  if (vec) k_u8_to_f32<true><<<cdiv(cdiv(n, 4), 256), 256, 0, st>>>(src, dst, n);
  else k_u8_to_f32<false><<<cdiv(cdiv(n, 4), 256), 256, 0, st>>>(src, dst, n);
  return cudaGetLastError();
}
cudaError_t launch_f32_to_u8(const float* src, uint8_t* dst, int64_t n, cudaStream_t st) {
  const bool vec = ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 3) == 0;
  if (vec) k_f32_to_u8<true><<<cdiv(cdiv(n, 4), 256), 256, 0, st>>>(src, dst, n);
  else k_f32_to_u8<false><<<cdiv(cdiv(n, 4), 256), 256, 0, st>>>(src, dst, n);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// feature_extractor.py:119  cfeat_conv_0: 3 -> 64, 3x3 SAME + bias + LeakyReLU, fp32 math.
// 8 threads per pixel (8 output channels each); 32 pixels per 256-thread block.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_conv0_c3(const float* __restrict__ img, int B, int H, int W,
                                                  const float* __restrict__ w,
                                                  const float* __restrict__ bias,
                                                  sp_t* __restrict__ out_hi, sp_t* __restrict__ out_lo,
                                                  int out_C, int out_c_off) {
  __shared__ float ws[27 * 64];
  __shared__ float bs[64];
  for (int i = threadIdx.x; i < 27 * 64; i += 256) ws[i] = w[i];
  if (threadIdx.x < 64) bs[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const int64_t npix = (int64_t)B * H * W;
  int64_t p = (int64_t)blockIdx.x * 32 + (threadIdx.x >> 3);
  if (p >= npix) return;
  const int g = threadIdx.x & 7;
  int x = (int)(p % W);
  int64_t q = p / W;
  int y = (int)(q % H);
  int b = (int)(q / H);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    int yy = y + ky - 1;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      int xx = x + kx - 1;
      if (xx < 0 || xx >= W) continue;
      const float* ip = img + (((int64_t)b * H + yy) * W + xx) * 3;
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        float v = __ldg(ip + ci);
        const float* wr = ws + ((ky * 3 + kx) * 3 + ci) * 64 + g * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(v, wr[j], acc[j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = leaky(acc[j] + bs[g * 8 + j]);
  uint4 h, l;
  pack8(acc, h, l);
  int64_t o = p * out_C + out_c_off + g * 8;
  *reinterpret_cast<uint4*>(out_hi + o) = h;
  *reinterpret_cast<uint4*>(out_lo + o) = l;
}

// ------------------------------------------------------------------------------------------
// cfeat_conv_0 of the product path (feature_extractor.py:119-123: 3 -> 64, 3x3 SAME, bias, LeakyReLU) as a
// register-tiled fp32 direct convolution.  K = 27 is far too short for the tensor cores (the MMA version pads it
// to 9 taps x 32 channels and is bound by its epilogue and by the widened 32-channel image tensor it needs), so
// the layer runs on the FMA pipes straight from the fp32 image: 1,728 FMAs per thread against 54 input and 108
// broadcast weight loads from shared memory.
//   block = 4 warps on an 8 x 16 pixel tile; warp w owns output channels [16w, 16w + 16);
//   lane  = (row lane / 4, four consecutive pixels from column 4 * (lane % 4)); 4 x 16 accumulators per thread.
// Exact fp32 arithmetic (the reference's own precision); writes the split planes of the 64-channel output.
// ------------------------------------------------------------------------------------------
constexpr int kC0H = 8, kC0W = 16;
constexpr int kC0Tiles = 4;   // consecutive tiles along x per block: weights are staged once, the next tile's input patch is
                              // fetched into registers while the current one is computed (the block prologue -- 7 KB of
                              // weights + a global round trip for the patch -- cost as much as the 1,728 FMAs of one tile)
constexpr int kC0Patch = (kC0H + 2) * (kC0W + 2) * 3;           // 540 floats
constexpr int kC0PatchRegs = (kC0Patch + 127) / 128;            // 5 per thread
__device__ __forceinline__ float fe_patch_load(const float* __restrict__ img, int b, int H, int W, int y0, int x0, int i) {
  const int c = i % 3, px = (i / 3) % (kC0W + 2), py = i / (3 * (kC0W + 2));
  const int yy = y0 + py - 1, xx = x0 + px - 1;
  return (i < kC0Patch && yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(img + (((int64_t)b * H + yy) * W + xx) * 3 + c) : 0.f;
}
__global__ void __launch_bounds__(128) k_fe_conv0(const float* __restrict__ img, int H, int W,
                                                  const float* __restrict__ w, const float* __restrict__ bias,
                                                  sp_t* __restrict__ out_hi, sp_t* __restrict__ out_lo, int lo_skip,
                                                  float* __restrict__ pool_out) {
  __shared__ float4 ws[27 * 16];                            // [tap * 3 + ci][64 channels]
  __shared__ float bs[64];
  __shared__ float patch[kC0Patch];                         // zero outside the image == SAME padding
  const int tid = threadIdx.x;
  const int b = blockIdx.z, y0 = blockIdx.y * kC0H, xb = blockIdx.x * (kC0W * kC0Tiles);
  for (int i = tid; i < 27 * 16; i += 128) ws[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
  if (tid < 64) bs[tid] = bias[tid];
  float nxt[kC0PatchRegs];
#pragma unroll
  for (int j = 0; j < kC0PatchRegs; ++j) nxt[j] = fe_patch_load(img, b, H, W, y0, xb, tid + 128 * j);
  const int warp = tid >> 5, lane = tid & 31;
  const int r = lane >> 2, cx = (lane & 3) * 4;
  const int y = y0 + r;
#pragma unroll 1
  for (int tile = 0; tile < kC0Tiles; ++tile) {
    const int x0 = xb + tile * kC0W;
    if (x0 >= W) break;                                     // block-uniform
    __syncthreads();                                        // everyone finished reading the previous patch
#pragma unroll
    for (int j = 0; j < kC0PatchRegs; ++j)
      if (tid + 128 * j < kC0Patch) patch[tid + 128 * j] = nxt[j];
    __syncthreads();
    // util.py:38-44 fused: the 2x2/2 average pool of this image level (= the next pyramid level, the input of the
    // same conv one scale up) is taken from the patch that is already in shared memory; same summation order as
    // k_image_pool, so the pyramid is bit-identical to the stand-alone kernel's
    if (pool_out != nullptr && tid < (kC0H / 2) * (kC0W / 2) * 3) {
      const int c = tid % 3, qx = (tid / 3) % (kC0W / 2), qy = tid / (3 * (kC0W / 2));
      const int oy = (y0 >> 1) + qy, ox = (x0 >> 1) + qx;
      if (oy < (H >> 1) && ox < (W >> 1)) {
        const float* p0 = patch + ((2 * qy + 1) * (kC0W + 2) + 2 * qx + 1) * 3 + c;
        const float* p1 = p0 + (kC0W + 2) * 3;
        pool_out[(((int64_t)b * (H >> 1) + oy) * (W >> 1) + ox) * 3 + c] = (p0[0] + p0[3] + p1[0] + p1[3]) * 0.25f;
      }
    }
    if (tile + 1 < kC0Tiles && x0 + kC0W < W) {             // prefetch the next tile's patch (latency hidden by the FMAs)
#pragma unroll
      for (int j = 0; j < kC0PatchRegs; ++j) nxt[j] = fe_patch_load(img, b, H, W, y0, x0 + kC0W, tid + 128 * j);
    }
    float acc[4][16];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[p][j] = 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      float in[18];                                         // 6 pixels x 3 channels of input row r + ky
      const float* pr = patch + ((r + ky) * (kC0W + 2) + cx) * 3;
#pragma unroll
      for (int j = 0; j < 18; ++j) in[j] = pr[j];
#pragma unroll
      for (int kx = 0; kx < 3; ++kx)
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) {
          const float4* wk = ws + ((ky * 3 + kx) * 3 + ci) * 16 + warp * 4;
          const float4 w0 = wk[0], w1 = wk[1], w2 = wk[2], w3 = wk[3];
          const float wv[16] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w};
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            const float v = in[(p + kx) * 3 + ci];
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[p][j] = fmaf(v, wv[j], acc[p][j]);
          }
        }
    }
    if (y < H) {
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int x = x0 + cx + p;
        if (x < W) {
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = leaky(acc[p][j] + bs[warp * 16 + j]);
          const int64_t o = (((int64_t)b * H + y) * W + x) * 64 + warp * 16;
          if (lo_skip) pack_store16_hi(f, out_hi + o);
          else pack_store16(f, out_hi + o, out_lo + o);
        }
      }
    }
  }
}
cudaError_t launch_fe_conv0(const float* img, int B, int H, int W, const float* w, const float* bias, sp_t* out_hi,
                            sp_t* out_lo, bool lo_skip, float* pool_out, cudaStream_t st) {
  dim3 grid((W + kC0W * kC0Tiles - 1) / (kC0W * kC0Tiles), (H + kC0H - 1) / kC0H, B);
  k_fe_conv0<<<grid, 128, 0, st>>>(img, H, W, w, bias, out_hi, out_lo, lo_skip ? 1 : 0, pool_out);
  return cudaGetLastError();
}

cudaError_t launch_conv0_c3(const float* img, int B, int H, int W, const float* w,
                            const float* bias, sp_t* out_hi, sp_t* out_lo, int out_C,
                            int out_c_off, cudaStream_t st) {
  int64_t npix = (int64_t)B * H * W;
  k_conv0_c3<<<cdiv(npix, 32), 256, 0, st>>>(img, B, H, W, w, bias, out_hi, out_lo, out_C, out_c_off);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// im2col-lite for cfeat_conv_0 (tensor-core path): out[p][k] = img[p + tap(k)][ci(k)],
// k = (ky*3 + kx)*3 + ci for k < 27, zero for 27 <= k < 32 and outside the image (SAME padding).
// The 3 -> 64 conv then is a 1x1 tensor-core conv with one 32-channel K block.
// 4 threads per pixel, 8 channels (one 128-bit store per plane) each.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_im2col3x3(const float* __restrict__ img, int B, int H, int W,
                                                   sp_t* __restrict__ out_hi, sp_t* __restrict__ out_lo) {
  const int64_t n = (int64_t)B * H * W * 4;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int g = (int)(i & 3);
  const int64_t p = i >> 2;
  const int x = (int)(p % W);
  const int64_t q = p / W;
  const int y = (int)(q % H);
  const int b = (int)(q / H);
  float v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = g * 8 + j;
    float val = 0.f;
    if (k < 27) {
      const int tap = k / 3, ci = k - tap * 3;
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) val = __ldg(img + (((int64_t)b * H + yy) * W + xx) * 3 + ci);
    }
    v[j] = val;
  }
  uint4 h, l;
  pack8(v, h, l);
  *reinterpret_cast<uint4*>(out_hi + p * 32 + g * 8) = h;
  *reinterpret_cast<uint4*>(out_lo + p * 32 + g * 8) = l;
}

// [B][H][W][3] fp32 image -> first 8 channels of a [B][H][W][32] split tensor (channels 3..31 stay at
// their initial zero): the input of cfeat_conv_0 when it runs on the persistent 3x3 tensor-core kernel.
__global__ void __launch_bounds__(256) k_image_to_split32(const float* __restrict__ img, int64_t npix,
                                                          sp_t* __restrict__ out_hi, sp_t* __restrict__ out_lo) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  float v[8] = {__ldg(img + p * 3), __ldg(img + p * 3 + 1), __ldg(img + p * 3 + 2), 0.f, 0.f, 0.f, 0.f, 0.f};
  uint4 h, l;
  pack8(v, h, l);
  *reinterpret_cast<uint4*>(out_hi + p * 32) = h;
  *reinterpret_cast<uint4*>(out_lo + p * 32) = l;
}

cudaError_t launch_image_to_split32(const float* img, int B, int H, int W, sp_t* out_hi, sp_t* out_lo, cudaStream_t st) {
  int64_t npix = (int64_t)B * H * W;
  k_image_to_split32<<<cdiv(npix, 256), 256, 0, st>>>(img, npix, out_hi, out_lo);
  return cudaGetLastError();
}

cudaError_t launch_im2col3x3(const float* img, int B, int H, int W, sp_t* out_hi, sp_t* out_lo, cudaStream_t st) {
  int64_t n = (int64_t)B * H * W * 4;
  k_im2col3x3<<<cdiv(n, 256), 256, 0, st>>>(img, B, H, W, out_hi, out_lo);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// feature_extractor.py:138-146  avg-pool of a channel slice of a split tensor
// ------------------------------------------------------------------------------------------
__global__ void k_act_pool(const sp_t* __restrict__ in_hi, const sp_t* __restrict__ in_lo, int in_C,
                           int in_c_off, int B, int H, int W, int Cn, sp_t* __restrict__ out_hi,
                           sp_t* __restrict__ out_lo, int out_C) {
  const int Ho = H / 2, Wo = W / 2, G = Cn / 8;
  const int64_t n = (int64_t)B * Ho * Wo * G;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int g = (int)(i % G);
  int64_t p = i / G;
  int x = (int)(p % Wo);
  int64_t q = p / Wo;
  int y = (int)(q % Ho);
  int b = (int)(q / Ho);
  int64_t base = (((int64_t)b * H + 2 * y) * W + 2 * x) * in_C + in_c_off + g * 8;
  float a[8], t[8];
  unpack8(ldg16(in_hi + base), ldg16(in_lo + base), a);
  unpack8(ldg16(in_hi + base + in_C), ldg16(in_lo + base + in_C), t);
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] += t[j];
  base += (int64_t)W * in_C;
  unpack8(ldg16(in_hi + base), ldg16(in_lo + base), t);
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] += t[j];
  unpack8(ldg16(in_hi + base + in_C), ldg16(in_lo + base + in_C), t);
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (a[j] + t[j]) * 0.25f;
  uint4 h, l;
  pack8(a, h, l);
  int64_t o = p * out_C + g * 8;
  *reinterpret_cast<uint4*>(out_hi + o) = h;
  *reinterpret_cast<uint4*>(out_lo + o) = l;
}

cudaError_t launch_act_pool(const sp_t* in_hi, const sp_t* in_lo, int in_C, int in_c_off, int B,
                            int H, int W, int Cn, sp_t* out_hi, sp_t* out_lo, int out_C,
                            cudaStream_t st) {
  int64_t n = (int64_t)B * (H / 2) * (W / 2) * (Cn / 8);
  if (n == 0) return cudaSuccess;
  k_act_pool<<<cdiv(n, 256), 256, 0, st>>>(in_hi, in_lo, in_C, in_c_off, B, H, W, Cn, out_hi, out_lo,
                                          out_C);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// fusion.py:133  tf.image.resize(NEAREST_NEIGHBOR) of a split tensor to a fine grid that is not twice
// the coarse one.  TF2 index rule in fp32: src = min(floor((dst + 0.5) * (in / out)), in - 1); the
// scales are fp32 quotients computed by the caller.  One thread copies 8 channels of one pixel.
// ------------------------------------------------------------------------------------------
template <bool kHiOnly>
__global__ void __launch_bounds__(256) k_resize_nearest(const sp_t* __restrict__ in_hi, const sp_t* __restrict__ in_lo,
                                                        int Hc, int Wc, int C, sp_t* __restrict__ out_hi,
                                                        sp_t* __restrict__ out_lo, int Hf, int Wf, int64_t n,
                                                        float sy, float sx) {
  const int G = C >> 3;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int g = (int)(i % G);
  const int64_t p = i / G;
  const int x = (int)(p % Wf);
  const int64_t q = p / Wf;
  const int y = (int)(q % Hf);
  const int b = (int)(q / Hf);
  const int ys = min((int)floorf(((float)y + 0.5f) * sy), Hc - 1);
  const int xs = min((int)floorf(((float)x + 0.5f) * sx), Wc - 1);
  const int64_t src = (((int64_t)b * Hc + ys) * Wc + xs) * C + g * 8;
  const int64_t dst = p * C + g * 8;
  *reinterpret_cast<uint4*>(out_hi + dst) = ldg16(in_hi + src);
  if (!kHiOnly) *reinterpret_cast<uint4*>(out_lo + dst) = ldg16(in_lo + src);
}

cudaError_t launch_resize_nearest(const sp_t* in_hi, const sp_t* in_lo, int B, int Hc, int Wc, int C, sp_t* out_hi,
                                  sp_t* out_lo, int Hf, int Wf, bool hi_only, cudaStream_t st) {
  if (C % 8) return cudaErrorInvalidValue;
  const int64_t n = (int64_t)B * Hf * Wf * (C / 8);
  if (n == 0) return cudaSuccess;
  const float sy = (float)Hc / (float)Hf, sx = (float)Wc / (float)Wf;
  if (hi_only) k_resize_nearest<true><<<cdiv(n, 256), 256, 0, st>>>(in_hi, in_lo, Hc, Wc, C, out_hi, out_lo, Hf, Wf, n, sy, sx);
  else k_resize_nearest<false><<<cdiv(n, 256), 256, 0, st>>>(in_hi, in_lo, Hc, Wc, C, out_hi, out_lo, Hf, Wf, n, sy, sx);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Shared gather helpers.
// TF2 bilinear resize (half-pixel centres):  src = (dst + 0.5) * in/out - 0.5
// TFA dense_image_warp / interpolate_bilinear border rule: floor clamped to [0, size-2],
// alpha clamped to [0, 1]  (SURVEY.md section 8c rules 4 and 6).
// ------------------------------------------------------------------------------------------
struct ResizeTap {
  int lo, hi;
  float w;
};
__device__ __forceinline__ ResizeTap resize_tap(int dst, int in_size, float scale) {
  float src = ((float)dst + 0.5f) * scale - 0.5f;
  float fl = floorf(src);
  ResizeTap t;
  t.lo = max((int)fl, 0);
  t.hi = min((int)ceilf(src), in_size - 1);
  t.w = src - fl;
  return t;
}

// 2 * v_prev resized to (H, W) at pixel (y, x) of batch d; v_prev is [2][Hc][Wc][2].
__device__ __forceinline__ float2 upsampled_flow(const float* __restrict__ v_prev, int d, int Hc,
                                                 int Wc, int H, int W, int y, int x) {
  const float sy = (float)Hc / (float)H, sx = (float)Wc / (float)W;
  ResizeTap ty = resize_tap(y, Hc, sy), tx = resize_tap(x, Wc, sx);
  const float2* base = reinterpret_cast<const float2*>(v_prev) + (int64_t)d * Hc * Wc;
  float2 tl = __ldg(base + (int64_t)ty.lo * Wc + tx.lo), tr = __ldg(base + (int64_t)ty.lo * Wc + tx.hi);
  float2 bl = __ldg(base + (int64_t)ty.hi * Wc + tx.lo), br = __ldg(base + (int64_t)ty.hi * Wc + tx.hi);
  float2 r;
  {
    float a = 2.f * tl.x, b = 2.f * tr.x, c = 2.f * bl.x, e = 2.f * br.x;
    float top = a + (b - a) * tx.w, bot = c + (e - c) * tx.w;
    r.x = top + (bot - top) * ty.w;
  }
  {
    float a = 2.f * tl.y, b = 2.f * tr.y, c = 2.f * bl.y, e = 2.f * br.y;
    float top = a + (b - a) * tx.w, bot = c + (e - c) * tx.w;
    r.y = top + (bot - top) * ty.w;
  }
  return r;
}

struct WarpTap {
  int y0, x0;
  float ay, ax;
};
__device__ __forceinline__ WarpTap warp_tap(int y, int x, float fx, float fy, int H, int W) {
  float qy = (float)y + fy, qx = (float)x + fx;
  float fy0 = fminf(fmaxf(floorf(qy), 0.f), (float)(H - 2));
  float fx0 = fminf(fmaxf(floorf(qx), 0.f), (float)(W - 2));
  WarpTap t;
  t.y0 = (int)fy0;
  t.x0 = (int)fx0;
  t.ay = fminf(fmaxf(qy - fy0, 0.f), 1.f);
  t.ax = fminf(fmaxf(qx - fx0, 0.f), 1.f);
  return t;
}

__device__ __forceinline__ float lerp4(float tl, float tr, float bl, float br, float ax, float ay) {
  float top = ax * (tr - tl) + tl;
  float bot = ax * (br - bl) + bl;
  return ay * (bot - top) + top;
}

// gather 8 channels of a split tensor plane pair [H][W][C] (already offset to the batch)
__device__ __forceinline__ void gather8(const sp_t* __restrict__ hi, const sp_t* __restrict__ lo,
                                        int W, int C, int c, const WarpTap& t, float* out) {
  const int64_t o00 = ((int64_t)t.y0 * W + t.x0) * C + c;
  const sp_t* h0 = hi + o00;
  const sp_t* l0 = lo + o00;
  const int row = W * C;  // < 2^31 elements for every level
  float tl[8], tr[8], bl[8], br[8];
  unpack8(ldg16(h0), ldg16(l0), tl);
  unpack8(ldg16(h0 + C), ldg16(l0 + C), tr);
  unpack8(ldg16(h0 + row), ldg16(l0 + row), bl);
  unpack8(ldg16(h0 + row + C), ldg16(l0 + row + C), br);
#pragma unroll
  for (int j = 0; j < 8; ++j) out[j] = lerp4(tl[j], tr[j], bl[j], br[j], t.ax, t.ay);
}

// gather 16 channels with 256-bit loads (two taps at a time to bound the live registers)
__device__ __forceinline__ void gather16(const sp_t* __restrict__ hi, const sp_t* __restrict__ lo,
                                         int W, int C, int c, const WarpTap& t, float* out) {
  const int64_t o00 = ((int64_t)t.y0 * W + t.x0) * C + c;
  const sp_t* h0 = hi + o00;
  const sp_t* l0 = lo + o00;
  const int row = W * C;
  float a[16], b[16], top[16];
  load_unpack16(h0, l0, a);
  load_unpack16(h0 + C, l0 + C, b);
#pragma unroll
  for (int j = 0; j < 16; ++j) top[j] = t.ax * (b[j] - a[j]) + a[j];
  load_unpack16(h0 + row, l0 + row, a);
  load_unpack16(h0 + row + C, l0 + row + C, b);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float bot = t.ax * (b[j] - a[j]) + a[j];
    out[j] = t.ay * (bot - top[j]) + top[j];
  }
}

// hi-plane-only gather: for destinations whose only consumers are single-pass convs (they read the hi plane
// alone, so the source is taken at hi precision too and the lo planes are neither read nor written)
__device__ __forceinline__ void gather16_hi(const sp_t* __restrict__ hi, int W, int C, int c, const WarpTap& t,
                                            float* out) {
  const sp_t* h0 = hi + ((int64_t)t.y0 * W + t.x0) * C + c;
  const int row = W * C;
  float a[16], b[16], top[16];
  load_unpack16_hi(h0, a);
  load_unpack16_hi(h0 + C, b);
#pragma unroll
  for (int j = 0; j < 16; ++j) top[j] = t.ax * (b[j] - a[j]) + a[j];
  load_unpack16_hi(h0 + row, a);
  load_unpack16_hi(h0 + row + C, b);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float bot = t.ax * (b[j] - a[j]) + a[j];
    out[j] = t.ay * (bot - top[j]) + top[j];
  }
}

// ------------------------------------------------------------------------------------------
// pyramid_flow_estimator.py:154-157  flow upsample (x2 magnitude) fused with the feature warp
// ------------------------------------------------------------------------------------------
template <bool kHiOnly>
__global__ void __launch_bounds__(256) k_flow_warp(const float* __restrict__ v_prev, int Hc, int Wc,
                                                   const sp_t* __restrict__ feat_hi,
                                                   const sp_t* __restrict__ feat_lo, int H, int W, int C,
                                                   float* __restrict__ v_up, sp_t* __restrict__ warped_hi,
                                                   sp_t* __restrict__ warped_lo) {
  // Block = 8 x 4 pixel patch x one 64-channel chunk (8 threads per pixel): the bilinear footprints of
  // vertically adjacent output pixels share source rows, so a 2-D patch turns those re-reads into L1 hits.
  // Block = 8 x 8 pixel patch x one 64-channel chunk, 4 threads per pixel x 16 channels (256-bit accesses);
  // grid = (tiles_x, tiles_y, 2 * C/64): no integer divisions in the index math
  const int nchunk = C >> 6;
  const int d = blockIdx.z / nchunk;
  const int c = (blockIdx.z - d * nchunk) * 64 + (threadIdx.x & 3) * 16;
  const int x = blockIdx.x * 8 + ((threadIdx.x >> 2) & 7), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  const int64_t p = ((int64_t)d * H + y) * W + x;  // pixel index over [2][H][W]
  // the upsampled flow is computed once per pixel (by the pixel's first thread) and shared through smem
  __shared__ float2 sflow[64];
  const int pix = threadIdx.x >> 2;
  if ((threadIdx.x & 3) == 0 && x < W && y < H) sflow[pix] = upsampled_flow(v_prev, d, Hc, Wc, H, W, y, x);
  __syncthreads();
  if (x >= W || y >= H) return;
  const float2 f = sflow[pix];
  if (c == 0) reinterpret_cast<float2*>(v_up)[p] = f;
  WarpTap t = warp_tap(y, x, f.x, f.y, H, W);
  const int64_t src_off = (int64_t)(1 - d) * H * W * C;
  float o[16];
  if constexpr (kHiOnly) {
    gather16_hi(feat_hi + src_off, W, C, c, t, o);
    pack_store16_hi(o, warped_hi + p * C + c);
  } else {
    gather16(feat_hi + src_off, feat_lo + src_off, W, C, c, t, o);
    pack_store16(o, warped_hi + p * C + c, warped_lo + p * C + c);
  }
}

cudaError_t launch_flow_warp(const float* v_prev, int Hc, int Wc, const sp_t* feat_hi,
                             const sp_t* feat_lo, int H, int W, int C, float* v_up,
                             sp_t* warped_hi, sp_t* warped_lo, bool hi_only, cudaStream_t st) {
  dim3 grid((W + 7) / 8, (H + 7) / 8, 2 * (C / 64));
  if (hi_only) k_flow_warp<true><<<grid, 256, 0, st>>>(v_prev, Hc, Wc, feat_hi, feat_lo, H, W, C, v_up, warped_hi, warped_lo);
  else k_flow_warp<false><<<grid, 256, 0, st>>>(v_prev, Hc, Wc, feat_hi, feat_lo, H, W, C, v_up, warped_hi, warped_lo);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// interpolator.py:163-178  fusion-stage warps (flows scaled by 0.5)
// ------------------------------------------------------------------------------------------
template <bool kHiOnly>
__global__ void __launch_bounds__(256) k_fusion_warp(const float* __restrict__ v,
                                                     const sp_t* __restrict__ feat_hi,
                                                     const sp_t* __restrict__ feat_lo, int H, int W,
                                                     int C, sp_t* __restrict__ warped_hi,
                                                     sp_t* __restrict__ warped_lo) {
  // 8 x 8 pixel patch x 64-channel chunk per block, 16 channels per thread (see k_flow_warp)
  const int nchunk = C >> 6;
  const int k = blockIdx.z / nchunk;
  const int c = (blockIdx.z - k * nchunk) * 64 + (threadIdx.x & 3) * 16;
  const int x = blockIdx.x * 8 + ((threadIdx.x >> 2) & 7), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  const int64_t p = ((int64_t)k * H + y) * W + x;
  // image k is warped by 0.5 * v[1 - k]
  float2 f = __ldg(reinterpret_cast<const float2*>(v) + ((int64_t)(1 - k) * H + y) * W + x);
  WarpTap t = warp_tap(y, x, f.x * 0.5f, f.y * 0.5f, H, W);
  const int64_t src_off = (int64_t)k * H * W * C;
  float o[16];
  if constexpr (kHiOnly) {
    gather16_hi(feat_hi + src_off, W, C, c, t, o);
    pack_store16_hi(o, warped_hi + p * C + c);
  } else {
    gather16(feat_hi + src_off, feat_lo + src_off, W, C, c, t, o);
    pack_store16(o, warped_hi + p * C + c, warped_lo + p * C + c);
  }
}

cudaError_t launch_fusion_warp(const float* v, const sp_t* feat_hi, const sp_t* feat_lo, int H,
                               int W, int C, sp_t* warped_hi, sp_t* warped_lo, bool hi_only, cudaStream_t st) {
  dim3 grid((W + 7) / 8, (H + 7) / 8, 2 * (C / 64));
  if (hi_only) k_fusion_warp<true><<<grid, 256, 0, st>>>(v, feat_hi, feat_lo, H, W, C, warped_hi, warped_lo);
  else k_fusion_warp<false><<<grid, 256, 0, st>>>(v, feat_hi, feat_lo, H, W, C, warped_hi, warped_lo);
  return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_fusion_side(const float* __restrict__ v,
                                                     const float* __restrict__ img, int H, int W,
                                                     sp_t* __restrict__ side_hi,
                                                     sp_t* __restrict__ side_lo, int side_C) {
  const int64_t n = (int64_t)H * W;
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  int x = (int)(p % W), y = (int)(p / W);
  float o[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) o[j] = 0.f;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    float2 f = __ldg(reinterpret_cast<const float2*>(v) + ((int64_t)(1 - k) * H + y) * W + x);
    f.x *= 0.5f;
    f.y *= 0.5f;
    WarpTap t = warp_tap(y, x, f.x, f.y, H, W);
    const float* ib = img + (int64_t)k * H * W * 3;
    const float* p00 = ib + ((int64_t)t.y0 * W + t.x0) * 3;
    const float* p10 = p00 + (int64_t)W * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      o[k * 3 + c] = lerp4(__ldg(p00 + c), __ldg(p00 + 3 + c), __ldg(p10 + c), __ldg(p10 + 3 + c), t.ax, t.ay);
    // k = 0 used the backward flow (v[1]) -> channels 6,7 ; k = 1 the forward flow -> 8,9
    o[6 + 2 * k] = f.x;
    o[7 + 2 * k] = f.y;
  }
  uint4 h, l;
  pack8(o, h, l);
  int64_t oo = p * side_C;
  *reinterpret_cast<uint4*>(side_hi + oo) = h;
  *reinterpret_cast<uint4*>(side_lo + oo) = l;
  pack8(o + 8, h, l);
  *reinterpret_cast<uint4*>(side_hi + oo + 8) = h;
  *reinterpret_cast<uint4*>(side_lo + oo + 8) = l;
}

cudaError_t launch_fusion_side(const float* v, const float* img, int H, int W, sp_t* side_hi,
                               sp_t* side_lo, int side_C, cudaStream_t st) {
  int64_t n = (int64_t)H * W;
  k_fusion_side<<<cdiv(n, 256), 256, 0, st>>>(v, img, H, W, side_hi, side_lo, side_C);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// pyramid_flow_estimator.py:77-83 + :161  flow head: 1x1 (nf -> nf/2, LReLU), 1x1 (-> 2), + v_up
// 32 pixels per 128-thread block; fp32 math.
// ------------------------------------------------------------------------------------------
constexpr int kHeadPix = 32;
__global__ void __launch_bounds__(128) k_flow_head(const sp_t* __restrict__ x_hi,
                                                   const sp_t* __restrict__ x_lo, int Cx, int nf,
                                                   int npix, const float* __restrict__ w3,
                                                   const float* __restrict__ b3,
                                                   const float* __restrict__ w4,
                                                   const float* __restrict__ b4,
                                                   const float* __restrict__ v_up,
                                                   float* __restrict__ residual, float* __restrict__ v) {
  extern __shared__ float smem[];
  const int J = nf / 2;
  float* xs = smem;                    // [kHeadPix][nf]
  float* hs = smem + kHeadPix * nf;    // [kHeadPix][J]
  const int64_t p0 = (int64_t)blockIdx.x * kHeadPix;
  const int G = nf / 8;
  for (int i = threadIdx.x; i < kHeadPix * G; i += 128) {
    int pp = i / G, g = i % G;
    float t[8];
    if (p0 + pp < npix) {
      int64_t o = (p0 + pp) * Cx + g * 8;
      unpack8(ldg16(x_hi + o), ldg16(x_lo + o), t);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) t[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) xs[pp * nf + g * 8 + j] = t[j];
  }
  __syncthreads();
  {
    const int j = threadIdx.x % J;
    const int groups = 128 / J > 0 ? 128 / J : 1;  // J <= 128
    const int pg = threadIdx.x / J;
    if (pg < groups) {
      for (int pp = pg; pp < kHeadPix; pp += groups) {
        float acc = 0.f;
        const float* xr = xs + pp * nf;
        for (int k = 0; k < nf; ++k) acc = fmaf(xr[k], __ldg(w3 + k * J + j), acc);
        hs[pp * J + j] = leaky(acc + __ldg(b3 + j));
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < kHeadPix * 2) {
    int pp = threadIdx.x >> 1, o = threadIdx.x & 1;
    if (p0 + pp < npix) {
      float acc = 0.f;
      const float* hr = hs + pp * J;
      for (int j = 0; j < J; ++j) acc = fmaf(hr[j], __ldg(w4 + j * 2 + o), acc);
      acc += __ldg(b4 + o);
      int64_t idx = (p0 + pp) * 2 + o;
      residual[idx] = acc;
      v[idx] = v_up ? acc + v_up[idx] : acc;
    }
  }
}

cudaError_t launch_flow_head(const sp_t* x_hi, const sp_t* x_lo, int Cx, int nf, int npix,
                             const float* w3, const float* b3, const float* w4, const float* b4,
                             const float* v_up, float* residual, float* v, cudaStream_t st) {
  size_t smem = (size_t)kHeadPix * (nf + nf / 2) * sizeof(float);
  k_flow_head<<<cdiv(npix, kHeadPix), 128, smem, st>>>(x_hi, x_lo, Cx, nf, npix, w3, b3, w4, b4, v_up,
                                                     residual, v);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// fusion.py:100-101,139  RGB head (1x1, 64 -> 3, linear) + crop
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rgb_head(const sp_t* __restrict__ x_hi,
                                                  const sp_t* __restrict__ x_lo, int Cx, int H, int W,
                                                  const float* __restrict__ w, const float* __restrict__ b,
                                                  float* __restrict__ out, int64_t out_pitch, int off_y,
                                                  int off_x, int out_h, int out_w) {
  __shared__ float ws[64 * 3 + 3];
  if (threadIdx.x < 64 * 3) ws[threadIdx.x] = w[threadIdx.x];
  if (threadIdx.x < 3) ws[192 + threadIdx.x] = b[threadIdx.x];
  __syncthreads();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)out_h * out_w) return;
  int ox = (int)(i % out_w), oy = (int)(i / out_w);
  int64_t p = (int64_t)(oy + off_y) * W + (ox + off_x);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    float t[8];
    unpack8(ldg16(x_hi + p * Cx + g * 8), ldg16(x_lo + p * Cx + g * 8), t);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float* wr = ws + (g * 8 + j) * 3;
      a0 = fmaf(t[j], wr[0], a0);
      a1 = fmaf(t[j], wr[1], a1);
      a2 = fmaf(t[j], wr[2], a2);
    }
  }
  float* o = out + (int64_t)oy * out_pitch + ox * 3;
  o[0] = a0 + ws[192];
  o[1] = a1 + ws[193];
  o[2] = a2 + ws[194];
}

cudaError_t launch_rgb_head(const sp_t* x_hi, const sp_t* x_lo, int Cx, int H, int W,
                            const float* w, const float* b, float* out, int64_t out_pitch,
                            int off_y, int off_x, int out_h, int out_w, cudaStream_t st) {
  int64_t n = (int64_t)out_h * out_w;
  k_rgb_head<<<cdiv(n, 256), 256, 0, st>>>(x_hi, x_lo, Cx, H, W, w, b, out, out_pitch, off_y, off_x,
                                          out_h, out_w);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// debug: split slice -> fp32
// ------------------------------------------------------------------------------------------
__global__ void k_unsplit(const sp_t* __restrict__ hi, const sp_t* __restrict__ lo, int C, int c_off,
                          int Cn, int64_t npix, float* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * Cn) return;
  int c = (int)(i % Cn);
  int64_t p = i / Cn;
  int64_t o = p * C + c_off + c;
  out[i] = sp_to_float(hi[o]) + sp_to_float(lo[o]);
}

cudaError_t launch_unsplit(const sp_t* hi, const sp_t* lo, int C, int c_off, int Cn, int64_t npix,
                           float* out, cudaStream_t st) {
  int64_t n = npix * Cn;
  k_unsplit<<<cdiv(n, 256), 256, 0, st>>>(hi, lo, C, c_off, Cn, npix, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// CUDA-core validation conv (debug option conv_impl = 1): same ConvProblem, fp32 FMA on the
// reconstructed hi+lo operands.  64 pixels x 64 output channels per 256-thread block.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_conv_simt(const ConvProblem* __restrict__ prob) {
  const ConvProblem& P = *prob;
  __shared__ float As[16][64 + 1];
  __shared__ float Ws[16][64 + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t npix = (int64_t)P.B * P.H * P.W;
  const int64_t m0 = (int64_t)blockIdx.x * 64;
  const int n0 = blockIdx.y * 64;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // loader mapping: thread loads A element (m = tid / 4, kk = (tid % 4) * 4 .. +3)
  const int lm = tid >> 2, lk = (tid & 3) * 4;
  int64_t pm = m0 + lm;
  int px = 0, py = 0, pb = 0;
  const bool pm_ok = pm < npix;
  if (pm_ok) {
    px = (int)(pm % P.W);
    int64_t q = pm / P.W;
    py = (int)(q % P.H);
    pb = (int)(q / P.H);
  }
  int kb = 0;
  const int KC = P.kchunk;
  for (int s = 0; s < P.nsrc; ++s) {
    const ConvSrc& S = P.src[s];
    for (int ch = 0; ch < S.nchunk; ++ch) {
      for (int t = 0; t < P.ntaps; ++t, ++kb) {
        const int yy = py + P.tap_dy[t], xx = px + P.tap_dx[t];
        const bool ok = pm_ok && yy >= 0 && yy < P.H && xx >= 0 && xx < P.W;
        const int64_t abase = (((int64_t)(S.bswap ? P.B - 1 - pb : pb) * P.H + yy) * P.W + xx) * S.C + S.c_off + ch * KC;
        for (int k16 = 0; k16 < KC; k16 += 16) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float v = 0.f;
            if (ok) v = sp_to_float(S.hi[abase + k16 + lk + e]) + sp_to_float(S.lo[abase + k16 + lk + e]);
            As[lk + e][lm] = v;
          }
          {
            // W element (n = tid / 4, kk = (tid%4)*4..)
            const int n = n0 + lm;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float v = 0.f;
              if (n < P.cout) {
                int64_t wi = (int64_t)n * P.ktot + (int64_t)kb * KC + k16 + lk + e;
                v = sp_to_float(P.w_hi[wi]) + sp_to_float(P.w_lo[wi]);
              }
              Ws[lk + e][lm] = v;
            }
          }
          __syncthreads();
#pragma unroll
          for (int kk = 0; kk < 16; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Ws[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
          }
          __syncthreads();
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t m = m0 + ty * 4 + i;
    if (m >= npix) continue;
    int x = (int)(m % P.W);
    int64_t q = m / P.W;
    int y = (int)(q % P.H);
    int b = (int)(q / P.H);
    int64_t opix = ((int64_t)b * P.out_H + (y * P.out_sy + P.out_oy)) * P.out_W + (x * P.out_sx + P.out_ox);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= P.cout) continue;
      float v = acc[i][j] + P.bias[n];
      if (P.act) v = leaky(v);
      sp_t h, l;
      split2(v, h, l);
      int64_t o = opix * P.out_C + P.out_c_off + n;
      P.out_hi[o] = h;
      P.out_lo[o] = l;
    }
  }
}

cudaError_t launch_conv_simt(const ConvProblem* d_prob, const ConvProblem& h, cudaStream_t st) {
  int64_t npix = (int64_t)h.B * h.H * h.W;
  dim3 grid(cdiv(npix, 64), cdiv(h.cout, 64));
  k_conv_simt<<<grid, 256, 0, st>>>(d_prob);
  return cudaGetLastError();
}

}  // namespace film
