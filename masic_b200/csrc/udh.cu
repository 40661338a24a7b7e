// udh.cu — the pieces of the homography front-end that are not convolutions (SURVEY §8(f)#4).
//
// Reference (file:line):
//   coremasic/mywork/model.py:52-69    Block: conv3x3 + ReLU, conv3x3 + ReLU, MaxPool2d(2,2)   -> maxpool2 below
//   coremasic/mywork/model.py:82-92    fc: Flatten, Linear(128*16*16, 1024), ReLU, Linear(1024, 8) -> fc_rows_kernel
//   coremasic/mywork/test2_real.py:201-211 (= model.py:103-111 get_h):
//        corners -= corners[:, 0];  corners_hat = corners + delta
//        h = kornia.get_perspective_transform(corners, corners_hat);  h_matrix = torch.inverse(h)
//        h_matrix = h_adjust(H, W, pic_size, pic_size, h_matrix)        (test2_real.py:54-64)   -> homography_kernel
// The 3x3 convolutions of the net run on conv_tc.cu (tcgen05); everything here is memory- or latency-bound.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"

namespace {

// 2x2 max-pool over NHWC bf16, 8 channels (16 bytes) per thread.
__global__ void __launch_bounds__(256)
maxpool2_kernel(const uint4* __restrict__ in, int n, int h, int w, int c8, uint4* __restrict__ out, int f16) {
  const int ho = h >> 1, wo = w >> 1;
  const long total = (long)n * ho * wo * c8;
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % c8);
  long r = i / c8;
  const int x = (int)(r % wo); r /= wo;
  const int y = (int)(r % ho);
  const int img = (int)(r / ho);
  const uint4* p = in + (((long)img * h + 2 * y) * w + 2 * x) * c8 + c;
  const uint4 a = __ldg(p), b = __ldg(p + c8), cc = __ldg(p + (long)w * c8), d = __ldg(p + (long)w * c8 + c8);
  auto mx = [f16](uint32_t u, uint32_t v) -> uint32_t { return masic::max16x2(u, v, f16); };
  uint4 o;
  o.x = mx(mx(a.x, b.x), mx(cc.x, d.x));
  o.y = mx(mx(a.y, b.y), mx(cc.y, d.y));
  o.z = mx(mx(a.z, b.z), mx(cc.z, d.z));
  o.w = mx(mx(a.w, b.w), mx(cc.w, d.w));
  out[i] = o;
}

// out[b][r] = act(bias[r] + sum_k w[r][k] * x[b][k]) for a handful of batch rows: one block per output row, the weight
// row is read once (16-byte loads, coalesced) and multiplied against every batch row (x stays in L1/L2: K * 2 bytes).
// HBM-bound: rows * K * 2 bytes of weights per call.
template <int MAXB>
__global__ void __launch_bounds__(256)
fc_rows_kernel(const __nv_bfloat16* __restrict__ x, int xb_stride, const __nv_bfloat16* __restrict__ w,
               const float* __restrict__ bias, int batch, int K, int relu, float* __restrict__ out_f32,
               __nv_bfloat16* __restrict__ out_bf16, int out_stride, int f16) {
  const int r = blockIdx.x;
  const uint4* wr = reinterpret_cast<const uint4*>(w + (size_t)r * K);
  float acc[MAXB];
#pragma unroll
  for (int b = 0; b < MAXB; ++b) acc[b] = 0.0f;
  for (int k8 = threadIdx.x; k8 < K / 8; k8 += blockDim.x) {
    const uint4 wv = __ldg(wr + k8);
    const uint32_t* w2 = reinterpret_cast<const uint32_t*>(&wv);
#pragma unroll
    for (int b = 0; b < MAXB; ++b) {
      if (b < batch) {
        const uint4 xv = __ldg(reinterpret_cast<const uint4*>(x + (size_t)b * xb_stride) + k8);
        const uint32_t* x2 = reinterpret_cast<const uint32_t*>(&xv);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 a = masic::unpack16x2(w2[e], f16), c = masic::unpack16x2(x2[e], f16);
          acc[b] = fmaf(a.x, c.x, acc[b]);
          acc[b] = fmaf(a.y, c.y, acc[b]);
        }
      }
    }
  }
  __shared__ float red[MAXB][8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int b = 0; b < MAXB; ++b) {
    float v = acc[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[b][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x < MAXB && threadIdx.x < batch) {
    const int b = threadIdx.x;
    float v = bias ? bias[r] : 0.0f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) v += red[b][i];
    if (relu) v = fmaxf(v, 0.0f);
    if (out_f32) out_f32[(size_t)b * out_stride + r] = v;
    if (out_bf16) reinterpret_cast<uint16_t*>(out_bf16)[(size_t)b * out_stride + r] = masic::pack16(v, f16);
  }
}

// [rows][C*H*W] (torch Flatten of NCHW: column = c*HW + p) -> bf16 [rows][HW*C] (column = p*C + c, the order of an NHWC
// activation), so the FC reads the conv output where it lies.
__global__ void fc_pack_kernel(const float* __restrict__ w, int rows, int c, int hw, uint16_t* __restrict__ dst, int f16) {
  const long total = (long)rows * c * hw;
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cc = (int)(i % c);
  long r = i / c;
  const int p = (int)(r % hw);
  const long row = r / hw;
  dst[i] = masic::pack16(w[(row * c + cc) * hw + p], f16);
}

// One thread per stereo pair: 8x8 DLT (Gaussian elimination with partial pivoting, fp64), 3x3 inverse, h_adjust.
__global__ void homography_kernel(const float* __restrict__ corners, const float* __restrict__ delta, int batch,
                                  int shift, float sa, float ia, float sb, float ib, float* __restrict__ h_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  double A[8][9];
  const float* c = corners + b * 8;
  const float* d = delta + b * 8;
  const float x0 = shift ? c[0] : 0.0f, y0 = shift ? c[1] : 0.0f;
  for (int i = 0; i < 4; ++i) {
    // test2_real.py:203: corners - corners[:, 0]; :206: corners_hat = corners + delta (fp32 tensors in the reference)
    const float xs = c[2 * i] - x0, ys = c[2 * i + 1] - y0;
    const float us = xs + d[2 * i], vs = ys + d[2 * i + 1];
    const double x = xs, y = ys, u = us, v = vs;
    double* r0 = A[2 * i];
    double* r1 = A[2 * i + 1];
    r0[0] = x; r0[1] = y; r0[2] = 1; r0[3] = 0; r0[4] = 0; r0[5] = 0; r0[6] = -x * u; r0[7] = -y * u; r0[8] = u;
    r1[0] = 0; r1[1] = 0; r1[2] = 0; r1[3] = x; r1[4] = y; r1[5] = 1; r1[6] = -x * v; r1[7] = -y * v; r1[8] = v;
  }
  for (int col = 0; col < 8; ++col) {
    int piv = col;
    for (int r = col + 1; r < 8; ++r) if (fabs(A[r][col]) > fabs(A[piv][col])) piv = r;
    if (piv != col) for (int k = 0; k < 9; ++k) { const double t = A[col][k]; A[col][k] = A[piv][k]; A[piv][k] = t; }
    const double inv = 1.0 / A[col][col];
    for (int r = 0; r < 8; ++r) {
      if (r == col) continue;
      const double f = A[r][col] * inv;
      if (f != 0.0) for (int k = col; k < 9; ++k) A[r][k] -= f * A[col][k];
    }
  }
  double m[9];
  for (int i = 0; i < 8; ++i) m[i] = A[i][8] / A[i][i];
  m[8] = 1.0;
  // torch.inverse(h)
  const double a00 = m[0], a01 = m[1], a02 = m[2], a10 = m[3], a11 = m[4], a12 = m[5], a20 = m[6], a21 = m[7], a22 = m[8];
  const double c00 = a11 * a22 - a12 * a21, c01 = a02 * a21 - a01 * a22, c02 = a01 * a12 - a02 * a11;
  const double c10 = a12 * a20 - a10 * a22, c11 = a00 * a22 - a02 * a20, c12 = a02 * a10 - a00 * a12;
  const double c20 = a10 * a21 - a11 * a20, c21 = a01 * a20 - a00 * a21, c22 = a00 * a11 - a01 * a10;
  const double idet = 1.0 / (a00 * c00 + a01 * c10 + a02 * c20);
  float h[9] = {(float)(c00 * idet), (float)(c01 * idet), (float)(c02 * idet), (float)(c10 * idet), (float)(c11 * idet),
                (float)(c12 * idet), (float)(c20 * idet), (float)(c21 * idet), (float)(c22 * idet)};
  // h_adjust (test2_real.py:54-64), in the reference's order of fp32 in-place updates:
  //   row 0 *= a;  column 0 *= 1/a;  row 1 *= b;  column 1 *= 1/b
  for (int k = 0; k < 3; ++k) h[k] = sa * h[k];
  for (int r = 0; r < 3; ++r) h[3 * r] = ia * h[3 * r];
  for (int k = 0; k < 3; ++k) h[3 + k] = sb * h[3 + k];
  for (int r = 0; r < 3; ++r) h[3 * r + 1] = ib * h[3 * r + 1];
  for (int i = 0; i < 9; ++i) h_out[b * 9 + i] = h[i];
}

}  // namespace

extern "C" int masic_maxpool2_nhwc_bf16(const void* in, int n, int h, int w, int c_pitch, void* out, int f16,
                                        void* stream) {
  if (!in || !out || n <= 0 || h <= 0 || w <= 0 || (h & 1) || (w & 1) || c_pitch <= 0 || (c_pitch & 7)) return MASIC_EINVAL;
  const long total = (long)n * (h / 2) * (w / 2) * (c_pitch / 8);
  maxpool2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(in), n, h, w, c_pitch / 8, static_cast<uint4*>(out), f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_fc_pack_weights(const float* weight, int rows, int c, int hw, void* dst_bf16, int f16,
                                     void* stream) {
  if (!weight || !dst_bf16 || rows <= 0 || c <= 0 || hw <= 0) return MASIC_EINVAL;
  const long total = (long)rows * c * hw;
  fc_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      weight, rows, c, hw, static_cast<uint16_t*>(dst_bf16), f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_fc_bf16(const void* x_bf16, int x_batch_stride, const void* w_bf16, const float* bias, int batch,
                             int k, int rows, int relu, float* out_f32, void* out_bf16, int out_batch_stride,
                             int f16, void* stream) {
  if (!x_bf16 || !w_bf16 || batch <= 0 || batch > 8 || k <= 0 || (k & 7) || (x_batch_stride & 7) || rows <= 0 ||
      (!out_f32 && !out_bf16))
    return MASIC_EINVAL;
  fc_rows_kernel<8><<<rows, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x_bf16), x_batch_stride, static_cast<const __nv_bfloat16*>(w_bf16), bias, batch,
      k, relu, out_f32, static_cast<__nv_bfloat16*>(out_bf16), out_batch_stride, f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_homography_from_delta(const float* corners, const float* delta, int batch, int shift_corners,
                                           int img_h, int img_w, int pic_h, int pic_w, float* h_out, void* stream) {
  if (!corners || !delta || !h_out || batch <= 0 || img_h <= 0 || img_w <= 0 || pic_h <= 0 || pic_w <= 0)
    return MASIC_EINVAL;
  // a = orishapea / resizeshapea, b = orishapeb / resizeshapeb as Python floats (doubles), then fp32 tensor * scalar
  const double a = (double)img_h / (double)pic_h, b = (double)img_w / (double)pic_w;
  homography_kernel<<<(batch + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(
      corners, delta, batch, shift_corners, (float)a, (float)(1.0 / a), (float)b, (float)(1.0 / b), h_out);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------ homographies in the zero-padded frame
namespace {

// T . H . T^-1 with T the translation by (left, top), in fp64 with the products and sums rounded one at a time in a
// fixed order (no contraction), rounded once to fp32: the same bits as the float64 expression written out on the host.
__global__ void homography_pad_kernel(const float* __restrict__ h_in, int n, double top, double left,
                                      float* __restrict__ h_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  double m[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) m[i] = (double)h_in[9 * b + i];
  double c[3];                                            // column 2 of H . T^-1
#pragma unroll
  for (int r = 0; r < 3; ++r) c[r] = __dsub_rn(__dsub_rn(m[3 * r + 2], __dmul_rn(left, m[3 * r])), __dmul_rn(top, m[3 * r + 1]));
  const float o[9] = {
      (float)__dadd_rn(m[0], __dmul_rn(left, m[6])), (float)__dadd_rn(m[1], __dmul_rn(left, m[7])),
      (float)__dadd_rn(c[0], __dmul_rn(left, c[2])),
      (float)__dadd_rn(m[3], __dmul_rn(top, m[6])), (float)__dadd_rn(m[4], __dmul_rn(top, m[7])),
      (float)__dadd_rn(c[1], __dmul_rn(top, c[2])),
      (float)m[6], (float)m[7], (float)c[2]};
#pragma unroll
  for (int i = 0; i < 9; ++i) h_out[9 * b + i] = o[i];
}

}  // namespace

extern "C" int masic_homography_pad(const float* h_in, int n, int top, int left, float* h_out, void* stream) {
  if (!h_in || !h_out || n <= 0) return MASIC_EINVAL;
  homography_pad_kernel<<<(n + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(h_in, n, (double)top,
                                                                                       (double)left, h_out);
  return (int)cudaGetLastError();
}
