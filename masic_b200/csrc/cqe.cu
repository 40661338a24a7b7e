// cqe.cu — memory-bound glue kernels of the cross quality enhancement network `Independent_EN`
// (coremasic/mywork/MASIC.py:1436-1501; SURVEY §8(f)#1).  The 3x3 convolutions of its Enhancement_Blocks run on the
// tensor-core conv kernel (conv_tc.cu) with LeakyReLU and the residual adds fused into the epilogue; what is left is
// the mask-weighted blending of an image / feature map with the homography-warped map of the OTHER view:
//   MASIC.py:1470-1471   cat(x_other_warp * w[0], x_self * w[1])              3 + 3 channels, images (NCHW fp32)
//   MASIC.py:1479-1482   cat(out_self * w[1], warp(out_other, H) * w[0])      32 + 32 channels, features (NHWC bf16)
//   MASIC.py:1493-1496   x_hat2 = conv2(out) + identity
// kornia.warp_perspective = bilinear, zero padding, align_corners=True (same coordinate chain as image.cu).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"

namespace {

struct Bilin { int x0, y0; float w00, w01, w10, w11; bool in_x0, in_x1, in_y0, in_y1; };

__device__ __forceinline__ Bilin bilin_coords(const double* __restrict__ t, int x, int y, int h, int w, int ho, int wo) {
  const double xn = ((double)x / (double)(wo - 1) - 0.5) * 2.0;
  const double yn = ((double)y / (double)(ho - 1) - 0.5) * 2.0;
  const double q0 = xn * t[0] + yn * t[1] + t[2];
  const double q1 = xn * t[3] + yn * t[4] + t[5];
  const double q2 = xn * t[6] + yn * t[7] + t[8];
  const double den = fabs(q2) >= 0.25 ? q2 : q2 + 1e-8;
  const double sc = fabs(q2) > 1e-8 ? 1.0 / den : 1.0;
  const double ixd = ((q0 * sc + 1.0) / 2.0) * (double)(w - 1);
  const double iyd = ((q1 * sc + 1.0) / 2.0) * (double)(h - 1);
  const double fxd = floor(ixd), fyd = floor(iyd);
  const float ix = (float)(ixd - fxd), iy = (float)(iyd - fyd);
  Bilin b;
  const bool finite = fabs(ixd) < 1e9 && fabs(iyd) < 1e9;
  b.x0 = finite ? (int)fxd : -10; b.y0 = finite ? (int)fyd : -10;
  b.w00 = (1.0f - ix) * (1.0f - iy); b.w01 = ix * (1.0f - iy); b.w10 = (1.0f - ix) * iy; b.w11 = ix * iy;
  b.in_x0 = b.x0 >= 0 && b.x0 < w; b.in_x1 = b.x0 + 1 >= 0 && b.x0 + 1 < w;
  b.in_y0 = b.y0 >= 0 && b.y0 < h; b.in_y1 = b.y0 + 1 >= 0 && b.y0 + 1 < h;
  return b;
}

// out[p][0:3] = a[:, p] * w[0][p], out[p][3:6] = b[:, p] * w[1][p], out[p][6:16] = 0      (bf16, pitch 16)
__global__ void __launch_bounds__(256)
blend_images_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ wgt, int n,
                    long hw, __nv_bfloat16* __restrict__ out, int f16) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n * hw) return;
  const int bi = (int)(i / hw);
  const long p = i - bi * hw;
  const float w0 = wgt[((long)bi * 2) * hw + p], w1 = wgt[((long)bi * 2 + 1) * hw + p];
  float v[6];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    v[c] = a[((long)bi * 3 + c) * hw + p] * w0;
    v[3 + c] = b[((long)bi * 3 + c) * hw + p] * w1;
  }
  uint32_t q[8];
#pragma unroll
  for (int j = 0; j < 3; ++j) q[j] = masic::pack16x2(v[2 * j], v[2 * j + 1], f16);
#pragma unroll
  for (int j = 3; j < 8; ++j) q[j] = 0u;
  uint4* o = reinterpret_cast<uint4*>(out + i * 16);
  o[0] = make_uint4(q[0], q[1], q[2], q[3]);
  o[1] = make_uint4(q[4], q[5], q[6], q[7]);
}

// out[p][0:C] = self[p][0:C] * w[1][p];  out[p][C:2C] = bilinear(other, T)[p][0:C] * w[0][p]
// A warp owns 32 consecutive pixels.  Phase 1: lane i evaluates the fp64 coordinate chain of pixel i (all 32 lanes busy:
// with one owner lane per pixel group the fp64 pipe ran at 1/8 utilisation and bounded the kernel).  Phase 2: the warp
// walks the 32 x 2*groups (pixel, 8-channel group) items, 32 per step, with 16-byte loads / stores; a step's lanes
// cover whole pixels, so every access is a run of contiguous 16-byte pieces.  C multiple of 8, 2*groups divides 32.
__global__ void __launch_bounds__(256)
feature_fuse_kernel(const __nv_bfloat16* __restrict__ self, int self_pitch, const __nv_bfloat16* __restrict__ other,
                    int other_pitch, int C, const float* __restrict__ wgt, const double* __restrict__ T, int n, int h,
                    int w, __nv_bfloat16* __restrict__ out, int out_pitch, int f16) {
  const int groups = C / 8, per_px = 2 * groups;
  const int lg = 31 - __clz(per_px);
  const int lane = threadIdx.x & 31;
  const unsigned hw32 = (unsigned)h * (unsigned)w;
  const unsigned warp_px0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32u;
  if (warp_px0 >= hw32) return;
  const int bi = blockIdx.y;
  const long hw = hw32;
  // ---- phase 1: coordinates and the two blend weights of pixel warp_px0 + lane
  const unsigned my_px = warp_px0 + lane;
  Bilin b;
  b.x0 = b.y0 = -10; b.w00 = b.w01 = b.w10 = b.w11 = 0.0f; b.in_x0 = b.in_x1 = b.in_y0 = b.in_y1 = false;
  float w_self = 0.0f, w_other = 0.0f;
  if (my_px < hw32) {
    const int y = (int)(my_px / (unsigned)w), x = (int)(my_px - (unsigned)y * (unsigned)w);
    b = bilin_coords(T + bi * 9, x, y, h, w, h, w);
    w_other = __ldg(wgt + ((long)bi * 2) * hw + my_px);
    w_self = __ldg(wgt + ((long)bi * 2 + 1) * hw + my_px);
  }
  const uint32_t my_flags = (uint32_t)b.in_x0 | ((uint32_t)b.in_x1 << 1) | ((uint32_t)b.in_y0 << 2) | ((uint32_t)b.in_y1 << 3);
  auto unpack = [f16](uint4 u, float* f) {
    const uint32_t q[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 t = masic::unpack16x2(q[j], f16);
      f[2 * j] = t.x; f[2 * j + 1] = t.y;
    }
  };
  // ---- phase 2
  for (int it = 0; it < per_px; ++it) {
    const int item = it * 32 + lane;
    const int src = item >> lg, g = item & (per_px - 1);      // pixel (lane that holds its coordinates), channel group
    const int x0 = __shfl_sync(0xffffffffu, b.x0, src), y0 = __shfl_sync(0xffffffffu, b.y0, src);
    const float w00 = __shfl_sync(0xffffffffu, b.w00, src), w01 = __shfl_sync(0xffffffffu, b.w01, src);
    const float w10 = __shfl_sync(0xffffffffu, b.w10, src), w11 = __shfl_sync(0xffffffffu, b.w11, src);
    const uint32_t fl = __shfl_sync(0xffffffffu, my_flags, src);
    const float ws = __shfl_sync(0xffffffffu, w_self, src), wo = __shfl_sync(0xffffffffu, w_other, src);
    const unsigned px = warp_px0 + src;
    if (px >= hw32) continue;
    const long p = (long)bi * hw + px;
    float acc[8];
    float scale;
    if (g < groups) {
      scale = ws;
      unpack(__ldg(reinterpret_cast<const uint4*>(self + p * self_pitch + 8 * g)), acc);
    } else {
      scale = wo;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
      const __nv_bfloat16* base = other + (long)bi * hw * other_pitch + 8 * (g - groups);
      auto tap = [&](bool ok, int yy, int xx, float wt) {
        if (!ok) return;
        float f[8];
        unpack(__ldg(reinterpret_cast<const uint4*>(base + ((long)yy * w + xx) * other_pitch)), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j] * wt;
      };
      tap((fl & 4u) && (fl & 1u), y0, x0, w00);
      tap((fl & 4u) && (fl & 2u), y0, x0 + 1, w01);
      tap((fl & 8u) && (fl & 1u), y0 + 1, x0, w10);
      tap((fl & 8u) && (fl & 2u), y0 + 1, x0 + 1, w11);
    }
    uint32_t q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = masic::pack16x2(acc[2 * j] * scale, acc[2 * j + 1] * scale, f16);
    *reinterpret_cast<uint4*>(out + p * out_pitch + 8 * g) = make_uint4(q[0], q[1], q[2], q[3]);
  }
}

// ---- training: backward of the two blends.  The images and the other view's features reach them from the frozen codec
// or from EB1; the mask weights come from mask2weights_EN, so they get a gradient too.
// Backward of feature_fuse_kernel for one view, g = dL/d(fused):
//   d_self[p][0:C]   = g[p][0:C] * w1[p]                                                      (bf16, stored)
//   d_other[q][0:C] += tap weight(p, q) * w0[p] * g[p][C:2C] over the four bilinear taps q   (fp32, atomics)
//   dmw[p][0] = sum_c g[p][C+c] * warp(other)[p][c];  dmw[p][1] = sum_c g[p][c] * self[p][c]  (NHWC fp32, stored)
// A warp owns 32 consecutive pixels: lane i evaluates the coordinates of pixel i (as in the forward), then the warp walks
// the pixels with its lanes over the channels.
__global__ void __launch_bounds__(256)
feature_fuse_bwd_kernel(const __nv_bfloat16* __restrict__ g, int g_pitch, const __nv_bfloat16* __restrict__ self,
                        int self_pitch, const __nv_bfloat16* __restrict__ other, int other_pitch, int C,
                        const float* __restrict__ wgt, const double* __restrict__ T, int h, int w,
                        __nv_bfloat16* __restrict__ d_self, int ds_pitch, float* __restrict__ d_other, int do_pitch,
                        float* __restrict__ dmw) {
  const int lane = threadIdx.x & 31;
  const unsigned hw32 = (unsigned)h * (unsigned)w;
  const unsigned warp_px0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32u;
  if (warp_px0 >= hw32) return;
  const int bi = blockIdx.y;
  const long hw = hw32;
  const unsigned my_px = warp_px0 + lane;
  Bilin b;
  b.x0 = b.y0 = -10; b.w00 = b.w01 = b.w10 = b.w11 = 0.0f; b.in_x0 = b.in_x1 = b.in_y0 = b.in_y1 = false;
  float w_self = 0.0f, w_other = 0.0f;
  if (my_px < hw32) {
    const int y = (int)(my_px / (unsigned)w), x = (int)(my_px - (unsigned)y * (unsigned)w);
    b = bilin_coords(T + bi * 9, x, y, h, w, h, w);
    w_other = __ldg(wgt + ((long)bi * 2) * hw + my_px);
    w_self = __ldg(wgt + ((long)bi * 2 + 1) * hw + my_px);
  }
  const uint32_t my_flags = (uint32_t)b.in_x0 | ((uint32_t)b.in_x1 << 1) | ((uint32_t)b.in_y0 << 2) | ((uint32_t)b.in_y1 << 3);
  const int npx = (int)min(32u, hw32 - warp_px0);
  const long img = (long)bi * hw;
  for (int j = 0; j < npx; ++j) {
    const int x0 = __shfl_sync(0xffffffffu, b.x0, j), y0 = __shfl_sync(0xffffffffu, b.y0, j);
    const float w00 = __shfl_sync(0xffffffffu, b.w00, j), w01 = __shfl_sync(0xffffffffu, b.w01, j);
    const float w10 = __shfl_sync(0xffffffffu, b.w10, j), w11 = __shfl_sync(0xffffffffu, b.w11, j);
    const uint32_t fl = __shfl_sync(0xffffffffu, my_flags, j);
    const float ws = __shfl_sync(0xffffffffu, w_self, j), wo = __shfl_sync(0xffffffffu, w_other, j);
    const long p = img + warp_px0 + j;
    float s0 = 0.0f, s1 = 0.0f;
    for (int c = lane; c < C; c += 32) {
      const float gs = __bfloat162float(g[p * g_pitch + c]), go = __bfloat162float(g[p * g_pitch + C + c]);
      s1 += gs * __bfloat162float(self[p * self_pitch + c]);
      d_self[p * ds_pitch + c] = __float2bfloat16_rn(gs * ws);
      const float gw = go * wo;
      float warped = 0.0f;
      auto tap = [&](bool ok, int yy, int xx, float wt) {
        if (!ok) return;
        const long q = img + (long)yy * w + xx;
        warped += __bfloat162float(other[q * other_pitch + c]) * wt;
        atomicAdd(d_other + q * do_pitch + c, wt * gw);
      };
      tap((fl & 4u) && (fl & 1u), y0, x0, w00);
      tap((fl & 4u) && (fl & 2u), y0, x0 + 1, w01);
      tap((fl & 8u) && (fl & 1u), y0 + 1, x0, w10);
      tap((fl & 8u) && (fl & 2u), y0 + 1, x0 + 1, w11);
      s0 += go * warped;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if (lane == 0) { dmw[p * 2] = s0; dmw[p * 2 + 1] = s1; }
  }
}

// Backward of blend_images_kernel w.r.t. the mask weights only, g = dL/d(out) as fp32 NHWC (channels 0..5 read):
//   dmw[p][0] += sum_c g[p][c] * a[c][p];  dmw[p][1] += sum_c g[p][3+c] * b[c][p]
__global__ void __launch_bounds__(256)
blend_images_bwd_kernel(const float* __restrict__ g, int g_pitch, const float* __restrict__ a,
                        const float* __restrict__ b, int n, long hw, float* __restrict__ dmw) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n * hw) return;
  const int bi = (int)(i / hw);
  const long p = i - bi * hw;
  float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    s0 += g[i * g_pitch + c] * a[((long)bi * 3 + c) * hw + p];
    s1 += g[i * g_pitch + 3 + c] * b[((long)bi * 3 + c) * hw + p];
  }
  dmw[i * 2] += s0;
  dmw[i * 2 + 1] += s1;
}

// out_nchw[b][c][p] = conv_out_nhwc[b][p][c] + identity_nchw[b][c][p],  c < 3
__global__ void __launch_bounds__(256)
residual_image_kernel(const float* __restrict__ conv_out, int pitch, const float* __restrict__ identity, int n, long hw,
                      float* __restrict__ out) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n * hw) return;
  const int bi = (int)(i / hw);
  const long p = i - bi * hw;
  const float4 v = *reinterpret_cast<const float4*>(conv_out + i * pitch);
  const float vv[3] = {v.x, v.y, v.z};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const long o = ((long)bi * 3 + c) * hw + p;
    out[o] = vv[c] + identity[o];
  }
}

// ------------------------------------------------------------------ mask2weights_EN, fused (MASIC.py:1411-1434)
// conv3x3(1->2)+ReLU, conv3x3(2->4)+ReLU, conv3x3(4->4)+ReLU, conv3x3(4->2), softmax over the 2 channels, all at full
// resolution: one block walks a 32x16 output tile through shared memory (9x9 receptive field = halo 4), so the mask
// is read once and only the two weights are written (12 B / pixel instead of ~100 B / pixel for four launches).
// Every layer zero-pads ITS OWN input (padding=1), hence intermediate values outside the image are forced to zero.
constexpr int MW_TW = 32, MW_TH = 16;

template <int CIN, int COUT, bool RELU>
__device__ __forceinline__ void mw_layer(const float* __restrict__ in, int in_w, int in_h, float* __restrict__ out,
                                         const float* __restrict__ wt, const float* __restrict__ bias, int gy0, int gx0,
                                         int H, int W) {
  // in: [CIN][in_h][in_w] covering image rows gy0-1.. ; out: [COUT][in_h-2][in_w-2] covering rows gy0..
  const int ow = in_w - 2, oh = in_h - 2;
  for (int i = threadIdx.x; i < ow * oh; i += blockDim.x) {
    const int oy = i / ow, ox = i - oy * ow;
    const int gy = gy0 + oy, gx = gx0 + ox;
    float acc[COUT];
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc[co] = bias[co];
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float v = in[(ci * in_h + oy + ky) * in_w + ox + kx];
#pragma unroll
          for (int co = 0; co < COUT; ++co) acc[co] = fmaf(v, wt[((co * CIN + ci) * 3 + ky) * 3 + kx], acc[co]);
        }
    const bool inside = gy >= 0 && gy < H && gx >= 0 && gx < W;
#pragma unroll
    for (int co = 0; co < COUT; ++co) {
      float r = RELU ? fmaxf(acc[co], 0.0f) : acc[co];
      out[(co * oh + oy) * ow + ox] = inside ? r : 0.0f;
    }
  }
}

__global__ void __launch_bounds__(256, 2)
mask_weights_en_kernel(const float* __restrict__ mask, int H, int W, const float* __restrict__ w1,
                       const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                       const float* __restrict__ w3, const float* __restrict__ b3, const float* __restrict__ w4,
                       const float* __restrict__ b4, float* __restrict__ out) {
  constexpr int W0 = MW_TW + 8, H0 = MW_TH + 8, W1 = W0 - 2, H1 = H0 - 2, W2 = W1 - 2, H2 = H1 - 2, W3 = W2 - 2,
                H3 = H2 - 2;
  __shared__ float s0[H0 * W0];
  __shared__ float s1[2 * H1 * W1];
  __shared__ float s2[4 * H2 * W2];
  __shared__ float s3[4 * H3 * W3];
  __shared__ float sw[18 + 72 + 144 + 72], sb[2 + 4 + 4 + 2];
  const int tid = threadIdx.x;
  for (int i = tid; i < 306; i += 256) sw[i] = i < 18 ? w1[i] : (i < 90 ? w2[i - 18] : (i < 234 ? w3[i - 90] : w4[i - 234]));
  if (tid < 12) sb[tid] = tid < 2 ? b1[tid] : (tid < 6 ? b2[tid - 2] : (tid < 10 ? b3[tid - 6] : b4[tid - 10]));
  const int n = blockIdx.z, y0 = blockIdx.y * MW_TH, x0 = blockIdx.x * MW_TW;
  const float* m = mask + (long)n * H * W;
  for (int i = tid; i < H0 * W0; i += 256) {
    const int py = i / W0, px = i - py * W0;
    const int gy = y0 - 4 + py, gx = x0 - 4 + px;
    s0[i] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? __ldg(m + (long)gy * W + gx) : 0.0f;
  }
  __syncthreads();
  mw_layer<1, 2, true>(s0, W0, H0, s1, sw, sb, y0 - 3, x0 - 3, H, W);
  __syncthreads();
  mw_layer<2, 4, true>(s1, W1, H1, s2, sw + 18, sb + 2, y0 - 2, x0 - 2, H, W);
  __syncthreads();
  mw_layer<4, 4, true>(s2, W2, H2, s3, sw + 90, sb + 6, y0 - 1, x0 - 1, H, W);
  __syncthreads();
  // last layer + softmax over the two channels (MASIC.py:1431), straight to global memory
  for (int i = tid; i < MW_TW * MW_TH; i += 256) {
    const int oy = i / MW_TW, ox = i - oy * MW_TW;
    const int gy = y0 + oy, gx = x0 + ox;
    if (gy >= H || gx >= W) continue;
    float a0 = sb[10], a1 = sb[11];
#pragma unroll
    for (int ci = 0; ci < 4; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float v = s3[(ci * H3 + oy + ky) * W3 + ox + kx];
          a0 = fmaf(v, sw[234 + ((0 * 4 + ci) * 3 + ky) * 3 + kx], a0);
          a1 = fmaf(v, sw[234 + ((1 * 4 + ci) * 3 + ky) * 3 + kx], a1);
        }
    const float mx = fmaxf(a0, a1);
    const float e0 = expf(a0 - mx), e1 = expf(a1 - mx);
    const float inv = 1.0f / (e0 + e1);
    const long o = ((long)n * 2) * H * W + (long)gy * W + gx;
    out[o] = e0 * inv;
    out[o + (long)H * W] = e1 * inv;
  }
}

}  // namespace

#define S(stream) static_cast<cudaStream_t>(stream)

extern "C" int masic_cqe_blend_images(const float* a_nchw, const float* b_nchw, const float* weights_nchw2, int n, int h,
                                      int w, void* out_nhwc16_bf16, int f16, void* stream) {
  if (!a_nchw || !b_nchw || !weights_nchw2 || !out_nhwc16_bf16 || n <= 0 || h <= 0 || w <= 0) return MASIC_EINVAL;
  const long total = (long)n * h * w;
  blend_images_kernel<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(
      a_nchw, b_nchw, weights_nchw2, n, (long)h * w, static_cast<__nv_bfloat16*>(out_nhwc16_bf16), f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_cqe_feature_fuse(const void* self_bf16, int self_pitch, const void* other_bf16, int other_pitch,
                                      int c, const float* weights_nchw2, const double* t_prepared, int n, int h, int w,
                                      void* out_bf16, int out_pitch, int f16, void* stream) {
  if (!self_bf16 || !other_bf16 || !weights_nchw2 || !t_prepared || !out_bf16 || c <= 0 || (c % 8) || (32 % (c / 4)) ||
      (self_pitch % 8) ||
      (other_pitch % 8) || (out_pitch % 8) || out_pitch < 2 * c || h < 2 || w < 2)
    return MASIC_EINVAL;
  const unsigned px_per_block = 256;                         // 8 warps x 32 pixels
  feature_fuse_kernel<<<dim3(((unsigned)h * (unsigned)w + px_per_block - 1) / px_per_block, n), 256, 0, S(stream)>>>(
      static_cast<const __nv_bfloat16*>(self_bf16), self_pitch, static_cast<const __nv_bfloat16*>(other_bf16), other_pitch,
      c, weights_nchw2, t_prepared, n, h, w, static_cast<__nv_bfloat16*>(out_bf16), out_pitch, f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_cqe_feature_fuse_bwd(const void* g_bf16, int g_pitch, const void* self_bf16, int self_pitch,
                                          const void* other_bf16, int other_pitch, int c, const float* weights_nchw2,
                                          const double* t_prepared, int n, int h, int w, void* d_self_bf16,
                                          int d_self_pitch, float* d_other_f32, int d_other_pitch,
                                          float* dweights_nhwc2, void* stream) {
  if (!g_bf16 || !self_bf16 || !other_bf16 || !weights_nchw2 || !t_prepared || !d_self_bf16 || !d_other_f32 ||
      !dweights_nhwc2 || c <= 0 || n <= 0 || h < 2 || w < 2 || g_pitch < 2 * c || self_pitch < c || other_pitch < c ||
      d_self_pitch < c || d_other_pitch < c)
    return MASIC_EINVAL;
  const unsigned px_per_block = 256;                         // 8 warps x 32 pixels
  feature_fuse_bwd_kernel<<<dim3(((unsigned)h * (unsigned)w + px_per_block - 1) / px_per_block, n), 256, 0, S(stream)>>>(
      static_cast<const __nv_bfloat16*>(g_bf16), g_pitch, static_cast<const __nv_bfloat16*>(self_bf16), self_pitch,
      static_cast<const __nv_bfloat16*>(other_bf16), other_pitch, c, weights_nchw2, t_prepared, h, w,
      static_cast<__nv_bfloat16*>(d_self_bf16), d_self_pitch, d_other_f32, d_other_pitch, dweights_nhwc2);
  return (int)cudaGetLastError();
}

extern "C" int masic_cqe_blend_images_bwd(const float* g_nhwc, int g_pitch, const float* a_nchw, const float* b_nchw,
                                          int n, int h, int w, float* dweights_nhwc2, void* stream) {
  if (!g_nhwc || !a_nchw || !b_nchw || !dweights_nhwc2 || g_pitch < 6 || n <= 0 || h <= 0 || w <= 0) return MASIC_EINVAL;
  const long total = (long)n * h * w;
  blend_images_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(g_nhwc, g_pitch, a_nchw, b_nchw, n,
                                                                                  (long)h * w, dweights_nhwc2);
  return (int)cudaGetLastError();
}

extern "C" int masic_cqe_residual_image(const float* conv_out_nhwc, int pitch, const float* identity_nchw, int n, int h,
                                        int w, float* out_nchw, void* stream) {
  if (!conv_out_nhwc || !identity_nchw || !out_nchw || pitch < 4 || (pitch % 4) || n <= 0) return MASIC_EINVAL;
  const long total = (long)n * h * w;
  residual_image_kernel<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(conv_out_nhwc, pitch, identity_nchw, n,
                                                                                (long)h * w, out_nchw);
  return (int)cudaGetLastError();
}

extern "C" int masic_cqe_mask_weights(const float* mask_nchw1, int n, int h, int w, const float* const* weights4,
                                      const float* const* biases4, int kw, float* out_nchw2, void* stream) {
  if (!mask_nchw1 || !weights4 || !biases4 || !out_nchw2 || n <= 0 || h <= 0 || w <= 0) return MASIC_EINVAL;
  if (kw != 2) return MASIC_ENOSUP;           // mask2weights_EN is only instantiated with Kw = 2 (MASIC.py:1449)
  for (int i = 0; i < 4; ++i)
    if (!weights4[i] || !biases4[i]) return MASIC_EINVAL;
  dim3 grid((w + MW_TW - 1) / MW_TW, (h + MW_TH - 1) / MW_TH, n);
  mask_weights_en_kernel<<<grid, 256, 0, S(stream)>>>(mask_nchw1, h, w, weights4[0], biases4[0], weights4[1], biases4[1],
                                                      weights4[2], biases4[2], weights4[3], biases4[3], out_nchw2);
  return (int)cudaGetLastError();
}
