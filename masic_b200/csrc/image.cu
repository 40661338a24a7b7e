// image.cu — memory-bound image-resolution kernels (sm_100a): homography warp, validity
// masks, the small-channel convolutions around the codec, layout packs.
//
// Replaces (reference, file:line):
//   kornia.warp_perspective call sites       coremasic/mywork/MASIC.py:781,821,833
//   mask()                                   MASIC.py:627-649
//   mask2weights (4x conv3 s2 + softmax)     MASIC.py:472-506
//   Encoder2.pre_conv + pre_gdn              MASIC.py:559-560,573-574
//   Decoder2.after_gdn + after_conv          MASIC.py:599-600,615-616
//   the pixel interleave of ConvTranspose2d(128->3) when it runs as a sub-pixel GEMM
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"

namespace {
using masic::pack16;
using masic::pack16x2;

// write c (<= 8) fp32 values as one zero-padded NHWC bf16 pixel of `pitch` channels with 16-byte stores
__device__ __forceinline__ void store_pixel_bf16(__nv_bfloat16* o, const float* v, int c, int pitch, int f16) {
  float e[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = i < c ? v[i] : 0.0f;
  if ((f16 & MASIC_FMT_SPLIT) && 2 * c <= 8 && 2 * c <= pitch) {     // [hi(c) | lo(c)]: lo = x - float(hi)
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i < c) {
        const float hi = masic::unpack16(pack16(e[i], f16), f16);
        const float lo = e[i] - hi;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j == c + i) e[j] = lo;       // compile-time indices keep e[] in registers
      }
  }
  if ((pitch & 7) == 0) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] = pack16x2(e[2 * i], e[2 * i + 1], f16);
    uint4* o4 = reinterpret_cast<uint4*>(o);
    o4[0] = make_uint4(w[0], w[1], w[2], w[3]);
    for (int j = 1; j < pitch / 8; ++j) o4[j] = make_uint4(0u, 0u, 0u, 0u);
  } else {
    uint16_t* o16 = reinterpret_cast<uint16_t*>(o);
    for (int ch = 0; ch < pitch; ++ch) {
      float x = 0.0f;
#pragma unroll
      for (int j = 0; j < 8; ++j) if (j == ch) x = e[j];
      o16[ch] = pack16(x, f16);
    }
  }
}

// same for 8 values already zero beyond the `c` real channels
__device__ __forceinline__ void store_pixel8_bf16(__nv_bfloat16* o, const float (&v)[8], int c, int pitch, int f16) {
  store_pixel_bf16(o, v, c, pitch, f16);
}

// ------------------------------------------------------------------ homography warp
// T = inv(N_dst * M * inv(N_src)) with N(h,w) = [[2/(w-1),0,-1],[0,2/(h-1),-1],[0,0,1]]
// (kornia 0.5.0 normalize_homography); evaluated and stored in fp64.  With invert_m != 0
// the function first replaces M by inv(M) (the second warp of mask(), MASIC.py:644).
__global__ void warp_prepare_kernel(const float* __restrict__ M, int batch, int h, int w, int ho, int wo,
                                    int invert_m, double* __restrict__ T) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  double m[9], a[9], r[9];
  for (int i = 0; i < 9; ++i) m[i] = (double)M[b * 9 + i];
  auto inv3 = [](const double* s, double* d) {
    const double c0 = s[4] * s[8] - s[5] * s[7], c1 = s[5] * s[6] - s[3] * s[8], c2 = s[3] * s[7] - s[4] * s[6];
    const double det = s[0] * c0 + s[1] * c1 + s[2] * c2;
    const double id = 1.0 / det;
    d[0] = c0 * id; d[1] = (s[2] * s[7] - s[1] * s[8]) * id; d[2] = (s[1] * s[5] - s[2] * s[4]) * id;
    d[3] = c1 * id; d[4] = (s[0] * s[8] - s[2] * s[6]) * id; d[5] = (s[2] * s[3] - s[0] * s[5]) * id;
    d[6] = c2 * id; d[7] = (s[1] * s[6] - s[0] * s[7]) * id; d[8] = (s[0] * s[4] - s[1] * s[3]) * id;
  };
  if (invert_m) { inv3(m, a); for (int i = 0; i < 9; ++i) m[i] = a[i]; }
  const double sw = (w == 1) ? 1e-14 : (double)(w - 1), sh = (h == 1) ? 1e-14 : (double)(h - 1);
  const double dw = (wo == 1) ? 1e-14 : (double)(wo - 1), dh = (ho == 1) ? 1e-14 : (double)(ho - 1);
  // inv(N_src) = [[sw/2,0,sw/2],[0,sh/2,sh/2],[0,0,1]];  a = M * inv(N_src)
  for (int i = 0; i < 3; ++i) {
    a[i * 3 + 0] = m[i * 3 + 0] * (sw / 2);
    a[i * 3 + 1] = m[i * 3 + 1] * (sh / 2);
    a[i * 3 + 2] = m[i * 3 + 0] * (sw / 2) + m[i * 3 + 1] * (sh / 2) + m[i * 3 + 2];
  }
  // r = N_dst * a
  for (int j = 0; j < 3; ++j) {
    r[0 + j] = (2.0 / dw) * a[0 + j] - a[6 + j];
    r[3 + j] = (2.0 / dh) * a[3 + j] - a[6 + j];
    r[6 + j] = a[6 + j];
  }
  inv3(r, a);
  for (int i = 0; i < 9; ++i) T[b * 9 + i] = a[i];
}

// 1/d to full fp64 accuracy from the fp32 reciprocal and two Newton steps (24 -> 48 -> 96 bits): ~8 instructions
// instead of the ~50 of an IEEE fp64 division (three of those per pixel were a fifth of the warp kernel's time).
__device__ __forceinline__ double fast_rcp(double d) {
  double r = (double)__frcp_rn((float)d);
  r = r * (2.0 - d * r);
  return r * (2.0 - d * r);
}

// One thread per destination pixel, all channels.  src == nullptr: source is all ones
// (mask(), MASIC.py:636-638) so the kernel is write-only.
// Outputs (either may be null): NCHW fp32, and NHWC bf16 with `bf_pitch` channels (zero padded).
// CT > 0: channel count known at compile time (the hot calls warp 3-channel images and the 1-channel mask): the
// per-channel values stay in registers and the guards of the generic CT = 0 form (local-memory arrays, ~300
// instructions per pixel, issue-bound) disappear.
template <int CT>
__global__ void __launch_bounds__(256)
warp_kernel(const float* __restrict__ src, int n, int c_rt, int h, int w, int ho, int wo,
            const double* __restrict__ T, double inv_wo1, double inv_ho1, float* __restrict__ dst,
            __nv_bfloat16* __restrict__ dst_bf, int bf_pitch, int bf_row, int bf_xoff, int f16,
            uint16_t* __restrict__ dst2, int d2_pitch, int d2_row, int d2_xoff, int d2_coff, int d2_f16) {
  const int c = CT ? CT : c_rt;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int b = blockIdx.z;
  if (x >= wo) return;
  const double* t = T + b * 9;
  // The reference evaluates this chain in fp32, which at 2176 px carries ~1e-4 px of rounding
  // noise of its own; the coordinates are evaluated in fp64 here (exact to ~1e-12 px) and only
  // the bilinear blend runs in fp32.  create_meshgrid(normalized): (i / (n-1) - 0.5) * 2
  // inv_wo1 = 1/(wo-1), inv_ho1 = 1/(ho-1) in fp64 from the host
  const double xn = ((double)x * inv_wo1 - 0.5) * 2.0;
  const double yn = ((double)y * inv_ho1 - 0.5) * 2.0;
  const double q0 = xn * t[0] + yn * t[1] + t[2];
  const double q1 = xn * t[3] + yn * t[4] + t[5];
  const double q2 = xn * t[6] + yn * t[7] + t[8];
  // convert_points_from_homogeneous: scale = |z| > 1e-8 ? 1/(z + 1e-8) : 1.  In the reference's fp32
  // the +1e-8 is absorbed whenever |z| >= 0.25 (half an ulp); keep that behaviour.
  const double den = fabs(q2) >= 0.25 ? q2 : q2 + 1e-8;
  const double aden = fabs(den);
  const double sc = fabs(q2) > 1e-8 ? ((aden > 1e-30 && aden < 1e30) ? fast_rcp(den) : 1.0 / den) : 1.0;
  const double gx = q0 * sc, gy = q1 * sc;
  // F.grid_sample(bilinear, zeros, align_corners=True)
  const double ixd = ((gx + 1.0) / 2.0) * (double)(w - 1);
  const double iyd = ((gy + 1.0) / 2.0) * (double)(h - 1);
  const double fxd = floor(ixd), fyd = floor(iyd);
  const float ix = (float)(ixd - fxd), iy = (float)(iyd - fyd);     // fractional parts in [0, 1)
  const float fx = 0.0f, fy = 0.0f;
  const float wx1 = ix - fx, wx0 = (fx + 1.0f) - ix;
  const float wy1 = iy - fy, wy0 = (fy + 1.0f) - iy;
  const float w_nw = wx0 * wy0, w_ne = wx1 * wy0, w_sw = wx0 * wy1, w_se = wx1 * wy1;
  // guard the int conversion against far-away coordinates
  const bool finite = fabs(ixd) < 1e9 && fabs(iyd) < 1e9;
  const int x0 = finite ? (int)fxd : -10, y0 = finite ? (int)fyd : -10;
  const bool in_x0 = x0 >= 0 && x0 < w, in_x1 = x0 + 1 >= 0 && x0 + 1 < w;
  const bool in_y0 = y0 >= 0 && y0 < h, in_y1 = y0 + 1 >= 0 && y0 + 1 < h;
  // out-of-image taps read a clamped address with a zero weight, so the four loads of every channel are independent
  // and all in flight at once (the kernel was bound by the latency of loads serialised behind their bounds branches)
  const float k_nw = (in_y0 && in_x0) ? w_nw : 0.0f, k_ne = (in_y0 && in_x1) ? w_ne : 0.0f;
  const float k_sw = (in_y1 && in_x0) ? w_sw : 0.0f, k_se = (in_y1 && in_x1) ? w_se : 0.0f;
  const int xc0 = min(max(x0, 0), w - 1), xc1 = min(max(x0 + 1, 0), w - 1);
  const int yc0 = min(max(y0, 0), h - 1), yc1 = min(max(y0 + 1, 0), h - 1);
  const int o_nw = yc0 * w + xc0, o_ne = yc0 * w + xc1, o_sw = yc1 * w + xc0, o_se = yc1 * w + xc1;   // one plane < 2^31 elements
  constexpr int NV = CT ? CT : 8;
  float vals[8];
#pragma unroll
  for (int ch = 0; ch < NV; ++ch) {
    if (!CT && ch >= c) break;
    float v = 0.0f;
    if (src) {
      const float* s = src + ((long)(b * c + ch) * h) * w;
      const float a = __ldg(s + o_nw), bq = __ldg(s + o_ne), cq = __ldg(s + o_sw), d = __ldg(s + o_se);
      // same accumulation order as before: nw, ne, sw, se (a zero-weight tap adds +0)
      v = a * k_nw;
      v += bq * k_ne;
      v += cq * k_sw;
      v += d * k_se;
    } else {
      v = ((k_nw + k_ne) + k_sw) + k_se;
    }
    vals[ch] = v;
    if (dst) dst[((long)(b * c + ch) * ho + y) * wo + x] = v;
  }
  if (dst_bf) {
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) if (ch >= c) vals[ch] = 0.0f;
    store_pixel_bf16(dst_bf + ((long)(b * ho + y) * bf_row + x + bf_xoff) * bf_pitch, vals, c, bf_pitch, f16);
  }
  if (dst2) {        // second 16-bit NHWC copy: the c values at channel d2_coff of a shared pixel slot (plain format)
    uint16_t* o = dst2 + ((long)(b * ho + y) * d2_row + x + d2_xoff) * d2_pitch + d2_coff;
    if (c == 3 && (d2_coff & 3) == 0 && (d2_pitch & 3) == 0) {     // one aligned 8-byte store: [v0 v1 v2 0]
      *reinterpret_cast<uint2*>(o) = make_uint2(pack16x2(vals[0], vals[1], d2_f16), pack16x2(vals[2], 0.0f, d2_f16));
    } else {
#pragma unroll
      for (int ch = 0; ch < NV; ++ch) if (ch < c) o[ch] = pack16(vals[ch], d2_f16);
    }
  }
}

// The engine's hot configurations of the kernel above (C = 3 or 1, fp32 planes and / or the two 16-bit images the
// right view's encoder and the tensor-core after_conv read), with the same per-pixel arithmetic in the same order
// (bit-identical outputs) and a fraction of the instructions: the generic form spends ~325 issued instructions per
// pixel, most of them 64-bit address arithmetic repeated for every tap and plane and the per-thread set-up (nine fp64
// matrix loads, the row terms).  Here a thread walks WF_PPT pixels of one row (x = x0 + i * WF_BLK, so a warp still
// touches 32 consecutive pixels), keeps the row terms yn * t[1,4,7] + nothing else hoisted (the fused multiply-adds of
// the generic form are kept as they are), holds one base pointer per source plane / destination row and reaches every
// tap with one 32-bit multiply-add.  SPLIT: dst16 pixels are [hi(3) | lo(3) | 0 0] halves (MASIC_FMT_F16 |
// MASIC_FMT_SPLIT, 8-channel pitch); dst2 is the plain fp16 [v0 v1 v2 0] half of a shared 8-channel pixel.
constexpr int WF_BLK = 64, WF_PPT = 4;
template <int CT>
__global__ void __launch_bounds__(WF_BLK)
warp_fast_kernel(const float* __restrict__ src, int h, int w, int ho, int wo, const double* __restrict__ T,
                 double inv_wo1, double inv_ho1, float* __restrict__ dst, uint16_t* __restrict__ dst16, int bf_row,
                 int bf_xoff, uint16_t* __restrict__ dst2, int d2_row, int d2_xoff, int d2_coff,
                 float* __restrict__ dst_ones) {
  const int y = blockIdx.y, b = blockIdx.z;
  const int xb = blockIdx.x * (WF_BLK * WF_PPT) + threadIdx.x;
  if (xb >= wo) return;
  const double* t = T + b * 9;
  const double t0 = t[0], t1 = t[1], t2 = t[2], t3 = t[3], t4 = t[4], t5 = t[5], t6 = t[6], t7 = t[7], t8 = t[8];
  const double yn = ((double)y * inv_ho1 - 0.5) * 2.0;
  const double r0 = yn * t1, r1 = yn * t4, r2 = yn * t7;
  const double wm1 = (double)(w - 1), hm1 = (double)(h - 1);
  const size_t hw = (size_t)h * w;
  const size_t dplane = (size_t)ho * wo;
  // one pointer per source plane and per destination row, pinned in registers (the opaque asm keeps the compiler from
  // folding the plane offset back into every tap's 64-bit index arithmetic): a tap is then base + 4 * u32
  const float* sp[CT];
  float* dp[CT];
#pragma unroll
  for (int ch = 0; ch < CT; ++ch) {
    sp[ch] = src ? src + ((size_t)b * CT + ch) * hw : nullptr;
    dp[ch] = dst ? dst + (((size_t)b * CT + ch) * ho + y) * wo : nullptr;
    asm volatile("" : "+l"(sp[ch]), "+l"(dp[ch]));
  }
  uint16_t* o16 = dst16 ? dst16 + ((size_t)(b * ho + y) * bf_row + bf_xoff) * 8 : nullptr;
  uint16_t* o2 = dst2 ? dst2 + ((size_t)(b * ho + y) * d2_row + d2_xoff) * 8 + d2_coff : nullptr;
  float* o1 = dst_ones ? dst_ones + ((size_t)b * ho + y) * wo : nullptr;     // warp of the all-ones image, same T
#pragma unroll
  for (int i = 0; i < WF_PPT; ++i) {
    const int x = xb + i * WF_BLK;
    if (x >= wo) break;
    const double xn = ((double)x * inv_wo1 - 0.5) * 2.0;
    const double q0 = fma(xn, t0, r0) + t2;
    const double q1 = fma(xn, t3, r1) + t5;
    const double q2 = fma(xn, t6, r2) + t8;
    const double den = fabs(q2) >= 0.25 ? q2 : q2 + 1e-8;
    const double aden = fabs(den);
    const double sc = fabs(q2) > 1e-8 ? ((aden > 1e-30 && aden < 1e30) ? fast_rcp(den) : 1.0 / den) : 1.0;
    const double gx = q0 * sc, gy = q1 * sc;
    const double ixd = ((gx + 1.0) / 2.0) * wm1;
    const double iyd = ((gy + 1.0) / 2.0) * hm1;
    const double fxd = floor(ixd), fyd = floor(iyd);
    const float ix = (float)(ixd - fxd), iy = (float)(iyd - fyd);
    const float wx1 = ix - 0.0f, wx0 = (0.0f + 1.0f) - ix;
    const float wy1 = iy - 0.0f, wy0 = (0.0f + 1.0f) - iy;
    const float w_nw = wx0 * wy0, w_ne = wx1 * wy0, w_sw = wx0 * wy1, w_se = wx1 * wy1;
    const bool finite = fabs(ixd) < 1e9 && fabs(iyd) < 1e9;
    const int x0 = finite ? (int)fxd : -10, y0 = finite ? (int)fyd : -10;
    float k_nw = w_nw, k_ne = w_ne, k_sw = w_sw, k_se = w_se;
    unsigned o_nw, d_e = 1u, d_s = (unsigned)w;                 // ne = nw + d_e, sw = nw + d_s, se = nw + d_s + d_e
    if (x0 >= 0 && x0 + 1 < w && y0 >= 0 && y0 + 1 < h) {       // all four taps inside the image (nearly every pixel)
      o_nw = (unsigned)(y0 * w + x0);
    } else {                                                   // border: zero weight on a clamped address
      const bool in_x0 = x0 >= 0 && x0 < w, in_x1 = x0 + 1 >= 0 && x0 + 1 < w;
      const bool in_y0 = y0 >= 0 && y0 < h, in_y1 = y0 + 1 >= 0 && y0 + 1 < h;
      k_nw = (in_y0 && in_x0) ? w_nw : 0.0f; k_ne = (in_y0 && in_x1) ? w_ne : 0.0f;
      k_sw = (in_y1 && in_x0) ? w_sw : 0.0f; k_se = (in_y1 && in_x1) ? w_se : 0.0f;
      const int xc0 = min(max(x0, 0), w - 1), xc1 = min(max(x0 + 1, 0), w - 1);
      const int yc0 = min(max(y0, 0), h - 1), yc1 = min(max(y0 + 1, 0), h - 1);
      o_nw = (unsigned)(yc0 * w + xc0);
      d_e = (unsigned)(xc1 - xc0);
      d_s = (unsigned)((yc1 - yc0) * w);
    }
    if (o1) o1[(unsigned)x] = ((k_nw + k_ne) + k_sw) + k_se;
    float vals[CT];
#pragma unroll
    for (int ch = 0; ch < CT; ++ch) {
      float v;
      if (src) {
        const float* s = sp[ch] + o_nw;
        const float* s2 = s + d_s;
        const float a = __ldg(s), bq = __ldg(s + d_e), cq = __ldg(s2), d = __ldg(s2 + d_e);
        v = a * k_nw;
        v += bq * k_ne;
        v += cq * k_sw;
        v += d * k_se;
      } else {
        v = ((k_nw + k_ne) + k_sw) + k_se;
      }
      vals[ch] = v;
      if (dst) dp[ch][(unsigned)x] = v;
    }
    if (CT == 3) {
      if (o16) {          // [hi0 hi1 hi2 lo0 | lo1 lo2 0 0] as one 16-byte store
        float lo[3];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch)
          lo[ch] = vals[ch] - masic::unpack16(pack16(vals[ch], MASIC_FMT_F16), MASIC_FMT_F16);
        *reinterpret_cast<uint4*>(o16 + (unsigned)x * 8u) =
            make_uint4(pack16x2(vals[0], vals[1], MASIC_FMT_F16), pack16x2(vals[2], lo[0], MASIC_FMT_F16),
                       pack16x2(lo[1], lo[2], MASIC_FMT_F16), 0u);
      }
      if (o2)
        *reinterpret_cast<uint2*>(o2 + (unsigned)x * 8u) =
            make_uint2(pack16x2(vals[0], vals[1], MASIC_FMT_F16), pack16x2(vals[2], 0.0f, MASIC_FMT_F16));
    }
  }
}

// ------------------------------------------------------------------ small-channel direct conv (NCHW fp32)
constexpr int SC_MAX_CO = 8, SC_MAX_CI = 8;

// out = act(conv_k(cat(in0, in1))) [-> GDN over the c_out channels]; one thread per output pixel.
template <int KT>     // KT = 3: fully unrolled 3x3 taps (all 9 loads of a channel in flight); KT = 0: generic loops
__global__ void __launch_bounds__(128)
conv_small_kernel(const float* __restrict__ in0, int c0, const float* __restrict__ in1, int c1,
                  int n, int h, int w, const float* __restrict__ wt, int transposed_s1,
                  const float* __restrict__ bias, int c_out, int k, int stride, int act,
                  int gdn, const float* __restrict__ beta, const float* __restrict__ gamma, float beta_bound,
                  int ho, int wo, float* __restrict__ out, __nv_bfloat16* __restrict__ out_bf, int bf_pitch,
                  int bf_row, int bf_xoff, int f16) {
  __shared__ float s_w[SC_MAX_CO * SC_MAX_CI * 25];
  __shared__ float s_b[SC_MAX_CO], s_beta[SC_MAX_CO], s_gamma[SC_MAX_CO * SC_MAX_CO];
  const int cin = c0 + c1, kk = k * k;
  for (int i = threadIdx.x; i < c_out * cin * kk; i += blockDim.x) {
    const int tap = i % kk, ci = (i / kk) % cin, co = i / (kk * cin);
    float v;
    if (transposed_s1) {   // ConvTranspose2d(stride 1) weight (cin, cout, k, k) == flipped conv
      const int ky = k - 1 - tap / k, kx = k - 1 - tap % k;
      v = wt[((ci * c_out + co) * k + ky) * k + kx];
    } else {
      v = wt[i];
    }
    s_w[i] = v;
  }
  if (threadIdx.x < c_out) s_b[threadIdx.x] = bias ? bias[threadIdx.x] : 0.0f;
  if (gdn) {
    const float ped = 1.4551915228366852e-11f;   // 2^-36
    if (threadIdx.x < c_out) { const float b = fmaxf(beta[threadIdx.x], beta_bound); s_beta[threadIdx.x] = b * b - ped; }
    for (int i = threadIdx.x; i < c_out * c_out; i += blockDim.x) {
      const float g = fmaxf(gamma[i], 3.814697265625e-06f);
      s_gamma[i] = g * g - ped;
    }
  }
  __syncthreads();
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= wo) return;
  float acc[SC_MAX_CO];
#pragma unroll
  for (int co = 0; co < SC_MAX_CO; ++co) acc[co] = co < c_out ? s_b[co] : 0.0f;
  const int pad = k / 2;
  if (KT == 3) {
    for (int ci = 0; ci < cin; ++ci) {
      const float* src = ci < c0 ? in0 + ((long)(b * c0 + ci) * h) * w : in1 + ((long)(b * c1 + (ci - c0)) * h) * w;
      float v[9];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int iy = y * stride - 1 + ky, ix = x * stride - 1 + kx;
          v[ky * 3 + kx] = (iy >= 0 && iy < h && ix >= 0 && ix < w) ? __ldg(src + (long)iy * w + ix) : 0.0f;
        }
#pragma unroll
      for (int tp = 0; tp < 9; ++tp)
#pragma unroll
        for (int co = 0; co < SC_MAX_CO; ++co)
          if (co < c_out) acc[co] = fmaf(v[tp], s_w[(co * cin + ci) * 9 + tp], acc[co]);
    }
  } else {
  for (int ci = 0; ci < cin; ++ci) {
    const float* src = ci < c0 ? in0 + ((long)(b * c0 + ci) * h) * w : in1 + ((long)(b * c1 + (ci - c0)) * h) * w;
    for (int ky = 0; ky < k; ++ky) {
      const int iy = y * stride - pad + ky;
      if (iy < 0 || iy >= h) continue;
      for (int kx = 0; kx < k; ++kx) {
        const int ix = x * stride - pad + kx;
        if (ix < 0 || ix >= w) continue;
        const float v = __ldg(src + (long)iy * w + ix);
#pragma unroll
        for (int co = 0; co < SC_MAX_CO; ++co)
          if (co < c_out) acc[co] = fmaf(v, s_w[(co * cin + ci) * kk + ky * k + kx], acc[co]);
      }
    }
  }
  }
  if (act == MASIC_ACT_RELU) {
#pragma unroll
    for (int co = 0; co < SC_MAX_CO; ++co) acc[co] = fmaxf(acc[co], 0.0f);
  } else if (act == MASIC_ACT_LEAKY) {
#pragma unroll
    for (int co = 0; co < SC_MAX_CO; ++co) acc[co] = acc[co] > 0.0f ? acc[co] : 0.01f * acc[co];
  }
  if (gdn) {
    float o[SC_MAX_CO];
#pragma unroll
    for (int i = 0; i < SC_MAX_CO; ++i) {
      if (i >= c_out) { o[i] = 0.0f; continue; }
      float nrm = s_beta[i];
      for (int j = 0; j < c_out; ++j) nrm = fmaf(s_gamma[i * c_out + j], acc[j] * acc[j], nrm);
      o[i] = acc[i] * (gdn == MASIC_GDN_FWD ? rsqrtf(nrm) : sqrtf(nrm));
    }
#pragma unroll
    for (int i = 0; i < SC_MAX_CO; ++i) acc[i] = o[i];
  }
  if (out)
    for (int co = 0; co < c_out; ++co) out[((long)(b * c_out + co) * ho + y) * wo + x] = acc[co];
  if (out_bf) {
    store_pixel_bf16(out_bf + ((long)(b * ho + y) * bf_row + x + bf_xoff) * bf_pitch, acc, c_out, bf_pitch, f16);
  }
}

// ------------------------------------------------------------------ 6 -> 3, 5x5, stride 1 (pre_conv / after_conv)
// Shared-memory tiled: a block of 16 x 8 threads produces 128 x 8 output pixels from a (128+4) x (8+4) x 6
// input patch staged once; each thread owns 2 x 4 horizontally adjacent pixels x 3 output channels (24
// accumulators), so per (ci, ky) it issues 4 conflict-free LDS.128 of pixels + 4 LDS.128 of (broadcast) weights
// for 120 FMAs: FMA-bound, not LDS-bound.  HBM traffic: 24 B in + 12 B out per pixel.
constexpr int F_TW = 128, F_TH = 8, F_PW = F_TW + 8, F_PH = F_TH + 4;   // pitch padded to 136 floats

__global__ void __launch_bounds__(128)
conv5x5_6to3_kernel(const float* __restrict__ in0, const float* __restrict__ in1, int n, int h, int w,
                    const float* __restrict__ wt, int transposed_s1, const float* __restrict__ bias,
                    int gdn, const float* __restrict__ beta, const float* __restrict__ gamma, float beta_bound,
                    float* __restrict__ out, __nv_bfloat16* __restrict__ out_bf, int bf_pitch, int bf_row,
                    int bf_xoff, int f16) {
  __shared__ __align__(16) float s_in[6][F_PH][F_PW];
  __shared__ __align__(16) float s_w[6 * 5 * 16];      // [ci][ky][kx*3 + co], 15 used of 16
  __shared__ float s_b[3], s_beta[3], s_gamma[9];
  const int tid = threadIdx.y * 16 + threadIdx.x;
  for (int i = tid; i < 6 * 5 * 16; i += 128) {
    const int j = i & 15, ky = (i >> 4) % 5, ci = i / 80;
    float v = 0.0f;
    if (j < 15) {
      const int kx = j / 3, co = j % 3;
      if (transposed_s1) v = wt[((ci * 3 + co) * 5 + (4 - ky)) * 5 + (4 - kx)];   // flipped conv
      else v = wt[((co * 6 + ci) * 5 + ky) * 5 + kx];
    }
    s_w[i] = v;
  }
  if (tid < 3) s_b[tid] = bias ? bias[tid] : 0.0f;
  if (gdn) {
    const float ped = 1.4551915228366852e-11f;
    if (tid < 3) { const float b = fmaxf(beta[tid], beta_bound); s_beta[tid] = b * b - ped; }
    if (tid < 9) { const float g = fmaxf(gamma[tid], 3.814697265625e-06f); s_gamma[tid] = g * g - ped; }
  }
  const int b = blockIdx.z, y0 = blockIdx.y * F_TH, x0 = blockIdx.x * F_TW;
  // stage the patch with aligned float4 global loads; s_in column c holds image column x0 - 2 + c
  const bool vec_ok = (w & 3) == 0;
  // loads are issued five at a time before any of them is stored: the staging phase used to expose one global-load
  // latency per iteration (a quarter of the kernel's stall samples)
  constexpr int N_STAGE = 6 * F_PH * (F_PW / 4), STAGE_BATCH = 5;
  for (int i0 = tid; i0 < N_STAGE; i0 += 128 * STAGE_BATCH) {
    float4 v[STAGE_BATCH];
#pragma unroll
    for (int u = 0; u < STAGE_BATCH; ++u) {
      const int i = i0 + u * 128;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < N_STAGE) {
        const int q = i % (F_PW / 4), py = (i / (F_PW / 4)) % F_PH, ci = i / ((F_PW / 4) * F_PH);
        const int gy = y0 + py - 2, gx = x0 + 4 * q - 4;
        if (gy >= 0 && gy < h) {
          const float* src = (ci < 3 ? in0 + ((long)(b * 3 + ci) * h) * w : in1 + ((long)(b * 3 + ci - 3) * h) * w) + (long)gy * w;
          if (vec_ok && gx >= 0 && gx + 3 < w) {
            v[u] = __ldg(reinterpret_cast<const float4*>(src + gx));
          } else {
            if (gx >= 0 && gx < w) v[u].x = __ldg(src + gx);
            if (gx + 1 >= 0 && gx + 1 < w) v[u].y = __ldg(src + gx + 1);
            if (gx + 2 >= 0 && gx + 2 < w) v[u].z = __ldg(src + gx + 2);
            if (gx + 3 >= 0 && gx + 3 < w) v[u].w = __ldg(src + gx + 3);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < STAGE_BATCH; ++u) {
      const int i = i0 + u * 128;
      if (i < N_STAGE) {
        const int q = i % (F_PW / 4), py = (i / (F_PW / 4)) % F_PH, ci = i / ((F_PW / 4) * F_PH);
        const int c = 4 * q - 2;
        if (c >= 0) *reinterpret_cast<float2*>(&s_in[ci][py][c]) = make_float2(v[u].x, v[u].y);
        if (c + 2 < F_PW) *reinterpret_cast<float2*>(&s_in[ci][py][c + 2]) = make_float2(v[u].z, v[u].w);
      }
    }
  }
  __syncthreads();
  // thread (tx, ty): pixels 4tx..4tx+3 (group 0) and 64+4tx..64+4tx+3 (group 1) of row ty: every LDS.128 of a
  // quarter-warp covers 128 contiguous bytes (no bank conflicts)
  float acc[2][4][3];
#pragma unroll
  for (int g = 0; g < 2; ++g)
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int co = 0; co < 3; ++co) acc[g][p][co] = s_b[co];
  const int lx = threadIdx.x * 4, ly = threadIdx.y;
#pragma unroll 1
  for (int ci = 0; ci < 6; ++ci) {
#pragma unroll
    for (int ky = 0; ky < 5; ++ky) {
      const float4* wq = reinterpret_cast<const float4*>(&s_w[(ci * 5 + ky) * 16]);
      const float4 w0 = wq[0], w1 = wq[1], w2 = wq[2], w3 = wq[3];
      const float ww[16] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w};
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        // output pixel lx+64g+p, tap kx reads image column x0 + lx + 64g + p + kx - 2 = s_in column lx + 64g + p + kx
        const float4 a0 = *reinterpret_cast<const float4*>(&s_in[ci][ly + ky][lx + 64 * g]);
        const float4 a1 = *reinterpret_cast<const float4*>(&s_in[ci][ly + ky][lx + 64 * g + 4]);
        const float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int kx = 0; kx < 5; ++kx) {
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            const float x = v[p + kx];
            acc[g][p][0] = fmaf(x, ww[kx * 3 + 0], acc[g][p][0]);
            acc[g][p][1] = fmaf(x, ww[kx * 3 + 1], acc[g][p][1]);
            acc[g][p][2] = fmaf(x, ww[kx * 3 + 2], acc[g][p][2]);
          }
        }
      }
    }
  }
  const int oy = y0 + ly;
  if (oy >= h) return;
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    if (gdn) {
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const float s0 = acc[g][p][0] * acc[g][p][0], s1 = acc[g][p][1] * acc[g][p][1], s2 = acc[g][p][2] * acc[g][p][2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const float nrm = fmaf(s_gamma[i * 3 + 2], s2, fmaf(s_gamma[i * 3 + 1], s1, fmaf(s_gamma[i * 3], s0, s_beta[i])));
          acc[g][p][i] *= (gdn == MASIC_GDN_FWD) ? rsqrtf(nrm) : sqrtf(nrm);
        }
      }
    }
    const int ox = x0 + lx + 64 * g;
    if (out) {
#pragma unroll
      for (int co = 0; co < 3; ++co) {
        float* o = out + ((long)(b * 3 + co) * h + oy) * w + ox;
        if (ox + 3 < w && (w & 3) == 0) {
          *reinterpret_cast<float4*>(o) = make_float4(acc[g][0][co], acc[g][1][co], acc[g][2][co], acc[g][3][co]);
        } else {
          for (int p = 0; p < 4; ++p) if (ox + p < w) o[p] = acc[g][p][co];
        }
      }
    }
    if (out_bf) {
      for (int p = 0; p < 4; ++p) {
        if (ox + p >= w) break;
        const float v3[8] = {acc[g][p][0], acc[g][p][1], acc[g][p][2], 0.f, 0.f, 0.f, 0.f, 0.f};
        store_pixel_bf16(out_bf + ((long)(b * h + oy) * bf_row + ox + p + bf_xoff) * bf_pitch, v3, 3, bf_pitch, f16);
      }
    }
  }
}

// ------------------------------------------------------------------ sub-pixel output -> NCHW (+ IGDN over 3 ch)
// in: [N][H2][W2][pitch] fp32, channel (py*2+px)*3 + co ; out: (N,3,2*H2,2*W2)
__global__ void __launch_bounds__(256)
subpix_to_nchw_kernel(const float* __restrict__ in, int n, int h2, int w2, int pitch, int gdn,
                      const float* __restrict__ beta, const float* __restrict__ gamma, float beta_bound,
                      float* __restrict__ out, __nv_bfloat16* __restrict__ out_bf, int bf_pitch, int f16) {
  __shared__ float s_beta[3], s_gamma[9];
  if (gdn && threadIdx.x < 9) {
    const float ped = 1.4551915228366852e-11f;
    const float g = fmaxf(gamma[threadIdx.x], 3.814697265625e-06f);
    s_gamma[threadIdx.x] = g * g - ped;
    if (threadIdx.x < 3) { const float b = fmaxf(beta[threadIdx.x], beta_bound); s_beta[threadIdx.x] = b * b - ped; }
  }
  __syncthreads();
  const int r = blockIdx.x * blockDim.x + threadIdx.x, q = blockIdx.y, b = blockIdx.z;
  if (r >= w2) return;
  const float4* ip = reinterpret_cast<const float4*>(in + ((long)(b * h2 + q) * w2 + r) * pitch);
  float v[12];
  const float4 a0 = ip[0], a1 = ip[1], a2 = ip[2];
  v[0] = a0.x; v[1] = a0.y; v[2] = a0.z; v[3] = a0.w; v[4] = a1.x; v[5] = a1.y; v[6] = a1.z; v[7] = a1.w;
  v[8] = a2.x; v[9] = a2.y; v[10] = a2.z; v[11] = a2.w;
  const int H = 2 * h2, W = 2 * w2;
#pragma unroll
  for (int ph = 0; ph < 4; ++ph) {
    float x0 = v[ph * 3], x1 = v[ph * 3 + 1], x2 = v[ph * 3 + 2];
    if (gdn) {
      const float s0 = x0 * x0, s1 = x1 * x1, s2 = x2 * x2;
      const float n0 = fmaf(s_gamma[2], s2, fmaf(s_gamma[1], s1, fmaf(s_gamma[0], s0, s_beta[0])));
      const float n1 = fmaf(s_gamma[5], s2, fmaf(s_gamma[4], s1, fmaf(s_gamma[3], s0, s_beta[1])));
      const float n2 = fmaf(s_gamma[8], s2, fmaf(s_gamma[7], s1, fmaf(s_gamma[6], s0, s_beta[2])));
      if (gdn == MASIC_GDN_FWD) { x0 *= rsqrtf(n0); x1 *= rsqrtf(n1); x2 *= rsqrtf(n2); }
      else { x0 *= sqrtf(n0); x1 *= sqrtf(n1); x2 *= sqrtf(n2); }
    }
    const int oy = 2 * q + (ph >> 1), ox = 2 * r + (ph & 1);
    if (out) {
      out[((long)(b * 3 + 0) * H + oy) * W + ox] = x0;
      out[((long)(b * 3 + 1) * H + oy) * W + ox] = x1;
      out[((long)(b * 3 + 2) * H + oy) * W + ox] = x2;
    }
    if (out_bf) {
      const float v3[8] = {x0, x1, x2, 0.f, 0.f, 0.f, 0.f, 0.f};
      store_pixel_bf16(out_bf + ((long)(b * H + oy) * W + ox) * bf_pitch, v3, 3, bf_pitch, f16);
    }
  }
}

// softmax over c (<= 8) channels of an NCHW tensor -> NCHW and/or NHWC ([pix][c]) fp32
__global__ void __launch_bounds__(256)
softmax_channels_kernel(const float* __restrict__ in, int n, int c, int hw, float* __restrict__ out_nchw,
                        float* __restrict__ out_nhwc) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n * hw) return;
  const int b = (int)(i / hw), p = (int)(i % hw);
  float v[8], mx = -INFINITY, sum = 0.0f;
  for (int ch = 0; ch < c; ++ch) { v[ch] = in[((long)(b * c + ch)) * hw + p]; mx = fmaxf(mx, v[ch]); }
  for (int ch = 0; ch < c; ++ch) { v[ch] = expf(v[ch] - mx); sum += v[ch]; }
  for (int ch = 0; ch < c; ++ch) {
    const float o = v[ch] / sum;
    if (out_nchw) out_nchw[((long)(b * c + ch)) * hw + p] = o;
    if (out_nhwc) out_nhwc[i * c + ch] = o;
  }
}

// ------------------------------------------------------------------ mask2weights in ONE launch (MASIC.py:472-506)
// conv3x3 s2 (1->3) ReLU, conv3x3 s2 (3->6) ReLU, conv3x3 s2 (6->6) ReLU, conv3x3 s2 (6->3), softmax over the 3 outputs.
// A block produces 4 x 4 positions of the 1/16-resolution map; the intermediate maps it needs (9x9, 19x19, 39x39
// positions) live in shared memory.  Every layer zero-pads its OWN input, so intermediate values outside a layer's
// domain are forced to zero.  Accumulation order per output = conv_small_kernel's (bias; ci; ky; kx), so the result
// is bit-identical to the five separate launches.
constexpr int MW_T = 4, MW_K3 = 2 * MW_T + 1, MW_K2 = 2 * MW_K3 + 1, MW_K1 = 2 * MW_K2 + 1;

__global__ void __launch_bounds__(256)
mask2weights_fused_kernel(const float* __restrict__ mask, int h, int w, const float* __restrict__ w1,
                          const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                          const float* __restrict__ w3, const float* __restrict__ b3, const float* __restrict__ w4,
                          const float* __restrict__ b4, float* __restrict__ out_nchw, float* __restrict__ out_nhwc) {
  __shared__ float s_k1[3][MW_K1][MW_K1 + 1];
  __shared__ float s_k2[6][MW_K2][MW_K2 + 1];
  __shared__ float s_k3[6][MW_K3][MW_K3 + 1];
  __shared__ float s_k4[3][MW_T * MW_T];
  __shared__ float s_w1[27], s_b1[3], s_w2[162], s_b2[6], s_w3[324], s_b3[6], s_w4[162], s_b4[3];
  const int tid = threadIdx.x, b = blockIdx.z;
  for (int i = tid; i < 324; i += 256) {
    s_w3[i] = w3[i];
    if (i < 162) { s_w2[i] = w2[i]; s_w4[i] = w4[i]; }
    if (i < 27) s_w1[i] = w1[i];
    if (i < 6) { s_b2[i] = b2 ? b2[i] : 0.0f; s_b3[i] = b3 ? b3[i] : 0.0f; }
    if (i < 3) { s_b1[i] = b1 ? b1[i] : 0.0f; s_b4[i] = b4 ? b4[i] : 0.0f; }
  }
  const int h1 = (h + 1) / 2, w1d = (w + 1) / 2, h2 = (h1 + 1) / 2, w2d = (w1d + 1) / 2;
  const int h3 = (h2 + 1) / 2, w3d = (w2d + 1) / 2, h4 = (h3 + 1) / 2, w4d = (w3d + 1) / 2;
  const int y4_0 = blockIdx.y * MW_T, x4_0 = blockIdx.x * MW_T;
  const int y3_0 = 2 * y4_0 - 1, x3_0 = 2 * x4_0 - 1;
  const int y2_0 = 2 * y3_0 - 1, x2_0 = 2 * x3_0 - 1;
  const int y1_0 = 2 * y2_0 - 1, x1_0 = 2 * x2_0 - 1;
  const float* src = mask + (long)b * h * w;
  __syncthreads();
  // layer 1: mask (global) -> s_k1
  for (int i = tid; i < MW_K1 * MW_K1; i += 256) {
    const int ly = i / MW_K1, lx = i % MW_K1, gy = y1_0 + ly, gx = x1_0 + lx;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
    if (gy >= 0 && gy < h1 && gx >= 0 && gx < w1d) {
      a0 = s_b1[0]; a1 = s_b1[1]; a2 = s_b1[2];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int iy = 2 * gy - 1 + ky, ix = 2 * gx - 1 + kx;
          const float v = (iy >= 0 && iy < h && ix >= 0 && ix < w) ? __ldg(src + (long)iy * w + ix) : 0.0f;
          a0 = fmaf(v, s_w1[0 * 9 + ky * 3 + kx], a0);
          a1 = fmaf(v, s_w1[1 * 9 + ky * 3 + kx], a1);
          a2 = fmaf(v, s_w1[2 * 9 + ky * 3 + kx], a2);
        }
      a0 = fmaxf(a0, 0.0f); a1 = fmaxf(a1, 0.0f); a2 = fmaxf(a2, 0.0f);
    }
    s_k1[0][ly][lx] = a0; s_k1[1][ly][lx] = a1; s_k1[2][ly][lx] = a2;
  }
  __syncthreads();
  // layer 2: s_k1 (3 ch) -> s_k2 (6 ch); one (position, channel) per task
  for (int i = tid; i < 6 * MW_K2 * MW_K2; i += 256) {
    const int co = i / (MW_K2 * MW_K2), r = i % (MW_K2 * MW_K2), ly = r / MW_K2, lx = r % MW_K2;
    const int gy = y2_0 + ly, gx = x2_0 + lx;
    float a = 0.0f;
    if (gy >= 0 && gy < h2 && gx >= 0 && gx < w2d) {
      a = s_b2[co];
#pragma unroll
      for (int ci = 0; ci < 3; ++ci)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
            a = fmaf(s_k1[ci][2 * ly + ky][2 * lx + kx], s_w2[(co * 3 + ci) * 9 + ky * 3 + kx], a);
      a = fmaxf(a, 0.0f);
    }
    s_k2[co][ly][lx] = a;
  }
  __syncthreads();
  // layer 3: s_k2 (6 ch) -> s_k3 (6 ch)
  for (int i = tid; i < 6 * MW_K3 * MW_K3; i += 256) {
    const int co = i / (MW_K3 * MW_K3), r = i % (MW_K3 * MW_K3), ly = r / MW_K3, lx = r % MW_K3;
    const int gy = y3_0 + ly, gx = x3_0 + lx;
    float a = 0.0f;
    if (gy >= 0 && gy < h3 && gx >= 0 && gx < w3d) {
      a = s_b3[co];
#pragma unroll
      for (int ci = 0; ci < 6; ++ci)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
            a = fmaf(s_k2[ci][2 * ly + ky][2 * lx + kx], s_w3[(co * 6 + ci) * 9 + ky * 3 + kx], a);
      a = fmaxf(a, 0.0f);
    }
    s_k3[co][ly][lx] = a;
  }
  __syncthreads();
  // layer 4 (no activation): s_k3 (6 ch) -> 3 logits per position
  if (tid < 3 * MW_T * MW_T) {
    const int co = tid / (MW_T * MW_T), r = tid % (MW_T * MW_T), ly = r / MW_T, lx = r % MW_T;
    float a = s_b4[co];
#pragma unroll
    for (int ci = 0; ci < 6; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
          a = fmaf(s_k3[ci][2 * ly + ky][2 * lx + kx], s_w4[(co * 6 + ci) * 9 + ky * 3 + kx], a);
    s_k4[co][r] = a;
  }
  __syncthreads();
  if (tid < MW_T * MW_T) {
    const int gy = y4_0 + tid / MW_T, gx = x4_0 + tid % MW_T;
    if (gy < h4 && gx < w4d) {
      float v[3], mx = -INFINITY, sum = 0.0f;
      for (int ch = 0; ch < 3; ++ch) { v[ch] = s_k4[ch][tid]; mx = fmaxf(mx, v[ch]); }
      for (int ch = 0; ch < 3; ++ch) { v[ch] = expf(v[ch] - mx); sum += v[ch]; }
      const long p = (long)gy * w4d + gx, hw4 = (long)h4 * w4d;
      for (int ch = 0; ch < 3; ++ch) {
        const float o = v[ch] / sum;
        if (out_nchw) out_nchw[((long)b * 3 + ch) * hw4 + p] = o;
        if (out_nhwc) out_nhwc[((long)b * hw4 + p) * 3 + ch] = o;
      }
    }
  }
}

// NCHW fp32 (c <= 8 real channels) -> NHWC bf16 with `pitch` channels, zero padded
__global__ void __launch_bounds__(256)
nchw_to_nhwc_bf16_kernel(const float* __restrict__ in, int f16, int n, int c, int hw, __nv_bfloat16* __restrict__ out,
                         int pitch, int w, int row, int xoff) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;      // batch on blockIdx.y: 32-bit index arithmetic only
  const int b = blockIdx.y;
  if (p >= hw) return;
  float v[8];
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) v[ch] = ch < c ? __ldg(in + ((long)(b * c + ch)) * hw + p) : 0.0f;
  const int y = p / w, x = p - y * w;
  store_pixel8_bf16(out + (((long)b * (hw / w) + y) * row + x + xoff) * pitch, v, c, pitch, f16);
}

// same for 3-channel images with w % 4 == 0: four pixels per thread (three 16-byte loads, four 16-byte stores)
__global__ void __launch_bounds__(256)
nchw3_to_nhwc_x4_kernel(const float* __restrict__ in, int f16, int hw, __nv_bfloat16* __restrict__ out, int pitch, int w,
                        int row, int xoff) {
  const int p = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int b = blockIdx.y;
  if (p >= hw) return;
  const float* src = in + (long)b * 3 * hw + p;
  const float4 c0 = __ldg(reinterpret_cast<const float4*>(src));
  const float4 c1 = __ldg(reinterpret_cast<const float4*>(src + hw));
  const float4 c2 = __ldg(reinterpret_cast<const float4*>(src + 2 * (long)hw));
  const int y = p / w, x = p - y * w;
  __nv_bfloat16* o = out + (((long)b * (hw / w) + y) * row + x + xoff) * pitch;
  const float px[4][8] = {{c0.x, c1.x, c2.x, 0.f, 0.f, 0.f, 0.f, 0.f}, {c0.y, c1.y, c2.y, 0.f, 0.f, 0.f, 0.f, 0.f},
                          {c0.z, c1.z, c2.z, 0.f, 0.f, 0.f, 0.f, 0.f}, {c0.w, c1.w, c2.w, 0.f, 0.f, 0.f, 0.f, 0.f}};
#pragma unroll
  for (int i = 0; i < 4; ++i) store_pixel8_bf16(o + (long)i * pitch, px[i], 3, pitch, f16);
}

// uint8 image -> float32 in [0, 1]: torchvision's ToTensor (img.float().div(255)).  The 256 possible results are computed
// once per block with the IEEE division (bit-identical to the host) and looked up: the kernel is then a pure stream
// (16 bytes in, 64 bytes out per thread) instead of 16 divisions per thread.
__global__ void __launch_bounds__(256)
u8_to_unit_f32_kernel(const uint8_t* __restrict__ in, long n, float* __restrict__ out) {
  __shared__ float lut[256];
  lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
  __syncthreads();
  const long i = (blockIdx.x * (long)blockDim.x + threadIdx.x) * 16;
  if (i >= n) return;
  if (i + 16 <= n && ((reinterpret_cast<uintptr_t>(in + i) & 15) == 0)) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(in + i));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 o;
      o.x = lut[w[q] & 255u];
      o.y = lut[(w[q] >> 8) & 255u];
      o.z = lut[(w[q] >> 16) & 255u];
      o.w = lut[w[q] >> 24];
      reinterpret_cast<float4*>(out + i)[q] = o;
    }
  } else {
    for (long j = i; j < n && j < i + 16; ++j) out[j] = lut[in[j]];
  }
}

// generic tiled transpose between NHWC and NCHW fp32 (c arbitrary)
__global__ void __launch_bounds__(256)
nhwc_to_nchw_f32_kernel(const float* __restrict__ in, int c, int hw, int in_pitch, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int p = p0 + j, ch = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (p < hw && ch < c) ? in[((long)b * hw + p) * in_pitch + ch] : 0.0f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int ch = c0 + j, p = p0 + threadIdx.x;
    if (p < hw && ch < c) out[((long)(b * c + ch)) * hw + p] = tile[threadIdx.x][j];
  }
}

}  // namespace

extern "C" int masic_warp_prepare(const float* m_3x3, int batch, int h, int w, int h_out, int w_out,
                                  int invert_m, double* t_out, void* stream) {
  if (!m_3x3 || !t_out || batch <= 0) return MASIC_EINVAL;
  warp_prepare_kernel<<<(batch + 31) / 32, 32, 0, static_cast<cudaStream_t>(stream)>>>(
      m_3x3, batch, h, w, h_out, w_out, invert_m, t_out);
  return (int)cudaGetLastError();
}

extern "C" int masic_warp_perspective_fwd(const float* src, int n, int c, int h, int w, int h_out, int w_out,
                                          const double* t_prepared, float* dst_nchw, void* dst_nhwc_bf16,
                                          int bf_pitch, int bf_row_pixels, int bf_xoff, int f16, void* dst2_nhwc16,
                                          int d2_pitch, int d2_row_pixels, int d2_xoff, int d2_coff, int d2_f16,
                                          float* dst_ones_nchw, void* stream) {
  if (!t_prepared || n <= 0 || c <= 0 || c > 8 || (!dst_nchw && !dst_nhwc_bf16 && !dst2_nhwc16 && !dst_ones_nchw))
    return MASIC_EINVAL;
  if (bf_row_pixels == 0) { bf_row_pixels = w_out; bf_xoff = 0; }
  if (bf_row_pixels < w_out + bf_xoff || bf_xoff < 0) return MASIC_EINVAL;
  if (dst2_nhwc16 && (d2_pitch < d2_coff + c || d2_coff < 0 || d2_xoff < 0 || d2_row_pixels < w_out + d2_xoff))
    return MASIC_EINVAL;
  if (h_out < 2 || w_out < 2) return MASIC_ENOSUP;
  if ((long)h * w >= (1L << 31)) return MASIC_ENOSUP;
  // the engine's configurations: 3- or 1-channel images, 16-bit copies (if any) as fp16 hi|lo pixels of pitch 8 and
  // as the aligned plain-fp16 half of a shared 8-channel pixel
  const bool fmt16_ok = !dst_nhwc_bf16 || (c == 3 && bf_pitch == 8 && f16 == (MASIC_FMT_F16 | MASIC_FMT_SPLIT));
  const bool fmt2_ok = !dst2_nhwc16 || (c == 3 && d2_pitch == 8 && (d2_coff & 3) == 0 && (d2_f16 & 1) == 1);
  if ((c == 3 || c == 1) && fmt16_ok && fmt2_ok && (long)n * c * h * w < (1L << 40)) {
    dim3 fgrid((w_out + WF_BLK * WF_PPT - 1) / (WF_BLK * WF_PPT), h_out, n);
    auto fk = c == 3 ? warp_fast_kernel<3> : warp_fast_kernel<1>;
    fk<<<fgrid, WF_BLK, 0, static_cast<cudaStream_t>(stream)>>>(
        src, h, w, h_out, w_out, t_prepared, 1.0 / (double)(w_out - 1), 1.0 / (double)(h_out - 1), dst_nchw,
        static_cast<uint16_t*>(dst_nhwc_bf16), bf_row_pixels, bf_xoff, static_cast<uint16_t*>(dst2_nhwc16),
        d2_row_pixels, d2_xoff, d2_coff, dst_ones_nchw);
    return (int)cudaGetLastError();
  }
  dim3 grid((w_out + 255) / 256, h_out, n);
  if (dst_ones_nchw) {          // generic path: the mask is a second launch with the all-ones source
    warp_kernel<1><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        nullptr, n, 1, h, w, h_out, w_out, t_prepared, 1.0 / (double)(w_out - 1), 1.0 / (double)(h_out - 1),
        dst_ones_nchw, nullptr, 0, w_out, 0, 0, nullptr, 0, 0, 0, 0, 0);
    if (!dst_nchw && !dst_nhwc_bf16 && !dst2_nhwc16) return (int)cudaGetLastError();
  }
  auto kern = c == 3 ? warp_kernel<3> : (c == 1 ? warp_kernel<1> : warp_kernel<0>);
  kern<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, n, c, h, w, h_out, w_out, t_prepared, 1.0 / (double)(w_out - 1), 1.0 / (double)(h_out - 1), dst_nchw,
      static_cast<__nv_bfloat16*>(dst_nhwc_bf16), bf_pitch, bf_row_pixels, bf_xoff, f16,
      static_cast<uint16_t*>(dst2_nhwc16), d2_pitch, d2_row_pixels, d2_xoff, d2_coff, d2_f16 & 1);
  return (int)cudaGetLastError();
}

extern "C" int masic_conv_small_nchw(const float* in0, int c0, const float* in1, int c1, int n, int h,
                                     int w, const float* weight, int transposed_s1, const float* bias,
                                     int c_out, int ksize, int stride, int act, int gdn, const float* beta,
                                     const float* gamma, float beta_min, float* out_nchw,
                                     void* out_nhwc_bf16, int bf_pitch, int bf_row_pixels, int bf_xoff,
                                     int f16, void* stream) {
  if (!in0 || !weight || c_out <= 0 || c_out > SC_MAX_CO || c0 + c1 > SC_MAX_CI || c0 <= 0) return MASIC_EINVAL;
  if ((ksize != 3 && ksize != 5 && ksize != 1) || (stride != 1 && stride != 2)) return MASIC_EINVAL;
  if (c1 > 0 && !in1) return MASIC_EINVAL;
  if (gdn && (!beta || !gamma)) return MASIC_EINVAL;
  if (transposed_s1 && stride != 1) return MASIC_EINVAL;
  const int ho = (h + stride - 1) / stride, wo = (w + stride - 1) / stride;
  if (bf_row_pixels == 0) { bf_row_pixels = wo; bf_xoff = 0; }
  if (bf_row_pixels < wo + bf_xoff || bf_xoff < 0) return MASIC_EINVAL;
  if (ksize == 5 && stride == 1 && c0 == 3 && c1 == 3 && c_out == 3 && act == MASIC_ACT_NONE &&
      (bf_pitch % 2 == 0)) {
    dim3 fgrid((w + F_TW - 1) / F_TW, (h + F_TH - 1) / F_TH, n), fblock(16, 8);
    conv5x5_6to3_kernel<<<fgrid, fblock, 0, static_cast<cudaStream_t>(stream)>>>(
        in0, in1, n, h, w, weight, transposed_s1, bias, gdn, beta, gamma,
        sqrtf(beta_min + 1.4551915228366852e-11f), out_nchw, static_cast<__nv_bfloat16*>(out_nhwc_bf16),
        bf_pitch, bf_row_pixels, bf_xoff, f16);
    return (int)cudaGetLastError();
  }
  dim3 grid((wo + 127) / 128, ho, n);
  auto kern = (ksize == 3) ? conv_small_kernel<3> : conv_small_kernel<0>;
  kern<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      in0, c0, in1, c1, n, h, w, weight, transposed_s1, bias, c_out, ksize, stride, act, gdn, beta, gamma,
      sqrtf(beta_min + 1.4551915228366852e-11f), ho, wo, out_nchw,
      static_cast<__nv_bfloat16*>(out_nhwc_bf16), bf_pitch, bf_row_pixels, bf_xoff, f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_subpix_to_nchw(const float* in_nhwc, int n, int h2, int w2, int pitch, int gdn,
                                    const float* beta, const float* gamma, float beta_min, float* out_nchw,
                                    void* out_nhwc_bf16, int bf_pitch, int f16, void* stream) {
  if (!in_nhwc || pitch < 12 || pitch % 4 || n <= 0) return MASIC_EINVAL;
  if (gdn && (!beta || !gamma)) return MASIC_EINVAL;
  dim3 grid((w2 + 255) / 256, h2, n);
  subpix_to_nchw_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in_nhwc, n, h2, w2, pitch, gdn, beta, gamma, sqrtf(beta_min + 1.4551915228366852e-11f), out_nchw,
      static_cast<__nv_bfloat16*>(out_nhwc_bf16), bf_pitch, f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_softmax_channels(const float* in_nchw, int n, int c, int hw, float* out_nchw,
                                      float* out_nhwc, void* stream) {
  if (!in_nchw || c <= 0 || c > 8 || n <= 0 || hw <= 0) return MASIC_EINVAL;
  const long total = (long)n * hw;
  softmax_channels_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in_nchw, n, c, hw, out_nchw, out_nhwc);
  return (int)cudaGetLastError();
}

extern "C" int masic_mask2weights(const float* mask_nchw, int n, int h, int w, const float* w1, const float* b1,
                                  const float* w2, const float* b2, const float* w3, const float* b3, const float* w4,
                                  const float* b4, float* out_nchw, float* out_nhwc, void* stream) {
  if (!mask_nchw || !w1 || !w2 || !w3 || !w4 || n <= 0 || h <= 0 || w <= 0 || (!out_nchw && !out_nhwc)) return MASIC_EINVAL;
  int ho = h, wo = w;
  for (int i = 0; i < 4; ++i) { ho = (ho + 1) / 2; wo = (wo + 1) / 2; }
  dim3 grid((wo + MW_T - 1) / MW_T, (ho + MW_T - 1) / MW_T, n);
  mask2weights_fused_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(mask_nchw, h, w, w1, b1, w2, b2, w3, b3,
                                                                                 w4, b4, out_nchw, out_nhwc);
  return (int)cudaGetLastError();
}

extern "C" int masic_nchw_to_nhwc_bf16(const float* in_nchw, int n, int c, int h, int w, void* out, int pitch,
                                       int row_pixels, int xoff, int f16, void* stream) {
  if (!in_nchw || !out || c <= 0 || c > 8 || c > pitch || pitch > 64 || h <= 0 || w <= 0) return MASIC_EINVAL;
  if (row_pixels == 0) { row_pixels = w; xoff = 0; }
  if (row_pixels < w + xoff || xoff < 0) return MASIC_EINVAL;
  const int hw = h * w;
  if (c == 3 && (w & 3) == 0 && (pitch & 7) == 0 && (reinterpret_cast<uintptr_t>(in_nchw) & 15) == 0) {
    nchw3_to_nhwc_x4_kernel<<<dim3((hw / 4 + 255) / 256, n), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        in_nchw, f16, hw, static_cast<__nv_bfloat16*>(out), pitch, w, row_pixels, xoff);
    return (int)cudaGetLastError();
  }
  nchw_to_nhwc_bf16_kernel<<<dim3((hw + 255) / 256, n), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in_nchw, f16, n, c, hw, static_cast<__nv_bfloat16*>(out), pitch, w, row_pixels, xoff);
  return (int)cudaGetLastError();
}

extern "C" int masic_nhwc_to_nchw_f32(const float* in_nhwc, int n, int c, int hw, int in_pitch,
                                      float* out_nchw, void* stream) {
  if (!in_nhwc || !out_nchw || n <= 0 || c <= 0 || hw <= 0 || in_pitch < c) return MASIC_EINVAL;
  dim3 grid((hw + 31) / 32, (c + 31) / 32, n), block(32, 8);
  nhwc_to_nchw_f32_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(in_nhwc, c, hw, in_pitch,
                                                                               out_nchw);
  return (int)cudaGetLastError();
}

extern "C" int masic_u8_to_unit_f32(const uint8_t* in_u8, int64_t numel, float* out_f32, void* stream) {
  if (!in_u8 || !out_f32 || numel < 0) return MASIC_EINVAL;
  if (numel == 0) return MASIC_OK;
  if (reinterpret_cast<uintptr_t>(out_f32) & 15) return MASIC_EINVAL;
  const long threads = (numel + 15) / 16;
  u8_to_unit_f32_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in_u8, numel, out_f32);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------ zero padding to the codec's 64-multiple frame
namespace {

constexpr int PAD_BLK = 256;

// One thread per 4 consecutive output columns of one padded row (n, c, Hp, Wp): every output element is written exactly
// once, the zero border included, so a padded buffer needs no memset and stays valid across pairs of one padded size.
// Rows and columns inside the source window read (uint8: torchvision's ToTensor, x / 255 with the IEEE division, as
// masic_u8_to_unit_f32) and optionally also write the unpadded float32 image from the same pass.
template <bool U8, bool VEC>
__global__ void __launch_bounds__(PAD_BLK)
pad_image_kernel(const void* __restrict__ src, int h, int w, int hp, int wp, int top, int left, long n_rows,
                 float* __restrict__ dst, float* __restrict__ dst_unpadded) {
  __shared__ float lut[256];
  if (U8) {
    lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
    __syncthreads();
  }
  const int q_per_row = (wp + 3) / 4;
  const long t = blockIdx.x * (long)PAD_BLK + threadIdx.x;
  if (t >= n_rows * q_per_row) return;
  const long row = t / q_per_row;                         // (image, channel, padded y)
  const int x0 = (int)(t - row * q_per_row) * 4;
  const long plane = row / hp;
  const int sy = (int)(row - plane * hp) - top;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (sy >= 0 && sy < h) {
    const long s_row = (plane * h + sy) * (long)w;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int sx = x0 + i - left;
      if (sx >= 0 && sx < w) {
        v[i] = U8 ? lut[static_cast<const uint8_t*>(src)[s_row + sx]] : static_cast<const float*>(src)[s_row + sx];
        if (dst_unpadded) dst_unpadded[s_row + sx] = v[i];
      }
    }
  }
  float* o = dst + row * wp + x0;
  if (VEC) {
    *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (x0 + i < wp) o[i] = v[i];
  }
}

}  // namespace

extern "C" int masic_pad_image(const void* src, int src_u8, int n, int c, int h, int w, int hp, int wp, int top,
                               int left, float* dst, float* dst_unpadded, void* stream) {
  if (!src || !dst || n <= 0 || c <= 0 || h <= 0 || w <= 0 || top < 0 || left < 0 || hp < h + top || wp < w + left)
    return MASIC_EINVAL;
  const long n_rows = (long)n * c * hp;
  const long threads = n_rows * ((wp + 3) / 4);
  const bool vec = (wp & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  auto k = src_u8 ? (vec ? pad_image_kernel<true, true> : pad_image_kernel<true, false>)
                  : (vec ? pad_image_kernel<false, true> : pad_image_kernel<false, false>);
  k<<<(unsigned)((threads + PAD_BLK - 1) / PAD_BLK), PAD_BLK, 0, static_cast<cudaStream_t>(stream)>>>(
      src, h, w, hp, wp, top, left, n_rows, dst, dst_unpadded);
  return (int)cudaGetLastError();
}
