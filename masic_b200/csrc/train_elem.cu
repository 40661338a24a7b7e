// train_elem.cu — memory-bound element-wise kernels of the training step over NHWC bf16 activations /
// gradients ([pixels][pitch], a slice of C channels at offset coff), with the per-channel sums the bias /
// beta gradients need fused in (sm_100a).
//
// Replaces the autograd backward (coremasic/mywork/newtrain_codec_real.py:134, loss.backward()) of:
//   nn.ReLU / nn.LeakyReLU(0.01) after conv()/deconv()          MASIC.py:173-183, 338-376, 410-444, 678-691
//   the bias add of nn.Conv2d / nn.ConvTranspose2d              compressai/models/utils.py:128-146
//   GDN.forward                                                 compressai/layers/gdn.py:77-92
//   NonNegativeParametrizer + LowerBound gradient               compressai/ops/parametrizers.py:61-64, bound_ops.py:36-58
//   torch.abs / additive-noise quantisation of the latents      MASIC.py:184, 755, 794, 823
//   the mask-weighted concatenation                             MASIC.py:827
// and, for the forward pass in train() mode, GDN as separate steps (the pre-GDN activation and the norm
// are kept for the backward pass): x -> x^2, norm = gamma' x^2 + beta' (a 1x1 conv on the tensor cores), y = x rsqrt(norm).
//
// Thread mapping of every [pixels][channels] kernel: 32 lanes x 2 channels = 64 channels per warp row, 8 pixel rows
// per block step, PIX_PER_BLOCK pixels per block; per-channel sums go through shared memory and one atomicAdd per
// (block, channel).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/masic_b200.h"

namespace {

constexpr int PIX_PER_BLOCK = 128;

__device__ __forceinline__ float2 ld_bf2(const __nv_bfloat16* p) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}
__device__ __forceinline__ void st_bf2(__nv_bfloat16* p, float a, float b) {
  *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}

// block (32, 8); grid (ceil(C/64), ceil(npix/PIX_PER_BLOCK)).  F(pixel, channel) -> value pair to sum per channel.
template <class F>
__device__ __forceinline__ void colsum_driver(long npix, int C, float* __restrict__ colsum, F f) {
  __shared__ float red[8][64];
  const int c = blockIdx.x * 64 + threadIdx.x * 2;
  const long p0 = (long)blockIdx.y * PIX_PER_BLOCK;
  float s0 = 0.0f, s1 = 0.0f;
  if (c < C) {
    const long pe = min(npix, p0 + PIX_PER_BLOCK);
    for (long p = p0 + threadIdx.y; p < pe; p += 8) {
      const float2 v = f(p, c);
      s0 += v.x; s1 += v.y;
    }
  }
  if (colsum) {
    red[threadIdx.y][threadIdx.x * 2] = s0;
    red[threadIdx.y][threadIdx.x * 2 + 1] = s1;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
      float a = 0.0f, b = 0.0f;
#pragma unroll
      for (int r = 0; r < 8; ++r) { a += red[r][threadIdx.x * 2]; b += red[r][threadIdx.x * 2 + 1]; }
      atomicAdd(colsum + c, a);
      if (c + 1 < C) atomicAdd(colsum + c + 1, b);
    }
  }
}

// g *= act'(y) in place; colsum += sum_p g   (bias gradient)
__global__ void __launch_bounds__(256)
act_bwd_bias_kernel(__nv_bfloat16* __restrict__ g, int gpitch, int gcoff, const __nv_bfloat16* __restrict__ y,
                    int ypitch, int ycoff, int act, long npix, int C, float* __restrict__ colsum) {
  colsum_driver(npix, C, colsum, [&](long p, int c) {
    __nv_bfloat16* gp = g + p * gpitch + gcoff + c;
    float2 v = ld_bf2(gp);
    if (act != MASIC_ACT_NONE) {
      const float2 yy = ld_bf2(y + p * ypitch + ycoff + c);
      const float slope = act == MASIC_ACT_RELU ? 0.0f : 0.01f;
      v.x = yy.x > 0.0f ? v.x : v.x * slope;
      v.y = yy.y > 0.0f ? v.y : v.y * slope;
      st_bf2(gp, v.x, v.y);
      v = ld_bf2(gp);                         // sum what the dgrad / wgrad kernels will read
    }
    return v;
  });
}

// out-of-place: dst = g * act'(y); colsum += sum_p dst.  g is left as it is (a residual block's skip still reads it).
__global__ void __launch_bounds__(256)
act_bwd_bias_out_kernel(const __nv_bfloat16* __restrict__ g, int gpitch, int gcoff, const __nv_bfloat16* __restrict__ y,
                        int ypitch, int ycoff, int act, long npix, int C, __nv_bfloat16* __restrict__ dst, int dpitch,
                        int dcoff, float* __restrict__ colsum) {
  colsum_driver(npix, C, colsum, [&](long p, int c) {
    float2 v = ld_bf2(g + p * gpitch + gcoff + c);
    if (act != MASIC_ACT_NONE) {
      const float2 yy = ld_bf2(y + p * ypitch + ycoff + c);
      const float slope = act == MASIC_ACT_RELU ? 0.0f : 0.01f;
      v.x = yy.x > 0.0f ? v.x : v.x * slope;
      v.y = yy.y > 0.0f ? v.y : v.y * slope;
    }
    __nv_bfloat16* dp = dst + p * dpitch + dcoff + c;
    st_bf2(dp, v.x, v.y);
    return ld_bf2(dp);                        // sum what the dgrad / wgrad kernels will read
  });
}

// fp32 gradient variant (sigma/mu/logit gradients arrive as bf16 already; this one serves fp32 sources): colsum only
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ g, int gpitch, int gcoff, long npix, int C,
                   float* __restrict__ colsum) {
  colsum_driver(npix, C, colsum, [&](long p, int c) { return ld_bf2(g + p * gpitch + gcoff + c); });
}

__global__ void __launch_bounds__(256)
gdn_sq_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ sq, long n2) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= n2) return;
  const float2 v = ld_bf2(x + 2 * i);
  st_bf2(sq + 2 * i, v.x * v.x, v.y * v.y);
}

// y = x * rsqrt(n)  (inverse: x * sqrt(n)); x bf16, n fp32, same [pixels][C] shape
__global__ void __launch_bounds__(256)
gdn_apply_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ nrm, int inverse,
                 __nv_bfloat16* __restrict__ y, long n2) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= n2) return;
  const float2 v = ld_bf2(x + 2 * i);
  const float2 n = *reinterpret_cast<const float2*>(nrm + 2 * i);
  const float r0 = inverse ? sqrtf(n.x) : rsqrtf(n.x), r1 = inverse ? sqrtf(n.y) : rsqrtf(n.y);
  st_bf2(y + 2 * i, v.x * r0, v.y * r1);
}

// GDN backward, step a.  y = x n^(-1/2):  t = -1/2 g x n^(-3/2), u = g n^(-1/2)
//                 IGDN   y = x n^(+1/2):  t = +1/2 g x n^(-1/2), u = g n^(+1/2)
// t -> tbuf (bf16), u overwrites g (bf16), dbeta' += sum_p t
__global__ void __launch_bounds__(256)
gdn_bwd_a_kernel(__nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ x, const float* __restrict__ nrm,
                 int inverse, __nv_bfloat16* __restrict__ tbuf, long npix, int C, float* __restrict__ dbeta) {
  colsum_driver(npix, C, dbeta, [&](long p, int c) {
    const long o = p * C + c;
    const float2 gg = ld_bf2(g + o), xx = ld_bf2(x + o);
    const float2 n = *reinterpret_cast<const float2*>(nrm + o);
    float t0, t1, u0, u1;
    if (inverse) {
      const float r0 = rsqrtf(n.x), r1 = rsqrtf(n.y);
      t0 = 0.5f * gg.x * xx.x * r0; t1 = 0.5f * gg.y * xx.y * r1;
      u0 = gg.x * (n.x * r0); u1 = gg.y * (n.y * r1);
    } else {
      const float r0 = rsqrtf(n.x), r1 = rsqrtf(n.y);
      t0 = -0.5f * gg.x * xx.x * (r0 * r0 * r0); t1 = -0.5f * gg.y * xx.y * (r1 * r1 * r1);
      u0 = gg.x * r0; u1 = gg.y * r1;
    }
    st_bf2(tbuf + o, t0, t1);
    st_bf2(g + o, u0, u1);
    return ld_bf2(tbuf + o);
  });
}

// GDN backward, step b: dx = u + 2 x v  (v = gamma'^T t from the 1x1 tensor-core conv), written over u;
// dbias += sum_p dx  (bias of the conv that feeds the GDN)
__global__ void __launch_bounds__(256)
gdn_bwd_b_kernel(__nv_bfloat16* __restrict__ u, const __nv_bfloat16* __restrict__ x, const float* __restrict__ v,
                 long npix, int C, float* __restrict__ dbias) {
  colsum_driver(npix, C, dbias, [&](long p, int c) {
    const long o = p * C + c;
    const float2 uu = ld_bf2(u + o), xx = ld_bf2(x + o);
    const float2 vv = *reinterpret_cast<const float2*>(v + o);
    st_bf2(u + o, uu.x + 2.0f * xx.x * vv.x, uu.y + 2.0f * xx.y * vv.y);
    return ld_bf2(u + o);
  });
}

// stored-parameter gradients from the gradients of beta' / gamma' (parametrizers.py:61-64 + LowerBound rule):
//   p' = max(p, bound)^2 - pedestal ;  g_lb = dp' * 2 max(p, bound) ;  dp = g_lb if (p >= bound or g_lb < 0) else 0
__global__ void reparam_bwd_kernel(const float* __restrict__ dprime, const float* __restrict__ stored, int n,
                                   float bound, int accumulate, float* __restrict__ dstored) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float p = stored[i];
  const float g = dprime[i] * 2.0f * fmaxf(p, bound);
  const float r = (p >= bound || g < 0.0f) ? g : 0.0f;
  dstored[i] = accumulate ? dstored[i] + r : r;
}

// every reparam_bwd of a training step (15 GDN layers x {beta, gamma}) as ONE launch: blockIdx.y = job
struct ReparamJob { const float* dprime; const float* stored; float* dstored; int n; float bound; int accumulate; int pad; };
__global__ void reparam_bwd_batch_kernel(const ReparamJob* __restrict__ jobs) {
  const ReparamJob j = jobs[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < j.n; i += gridDim.x * blockDim.x) {
    const float p = j.stored[i];
    const float g = j.dprime[i] * 2.0f * fmaxf(p, j.bound);
    const float r = (p >= j.bound || g < 0.0f) ? g : 0.0f;
    j.dstored[i] = j.accumulate ? j.dstored[i] + r : r;
  }
}

// |y| and y + noise as bf16 NHWC copies of an fp32 NHWC latent [pixels][C]
__global__ void __launch_bounds__(256)
latent_prep_train_kernel(const float* __restrict__ y, const float* __restrict__ noise, long total, int C,
                         __nv_bfloat16* __restrict__ y_abs, int abs_pitch, __nv_bfloat16* __restrict__ y_noisy,
                         int noisy_pitch) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long p = i / C;
  const int c = (int)(i - p * C);
  const float v = y[i];
  if (y_abs) y_abs[p * abs_pitch + c] = __float2bfloat16_rn(fabsf(v));
  if (y_noisy) y_noisy[p * noisy_pitch + c] = __float2bfloat16_rn(v + noise[i]);
}

// dy = dy_lik + d_dec + d_ctx + sign(y) d_abs   (any source may be NULL) -> bf16 [pixels][C]
__global__ void __launch_bounds__(256)
latent_merge_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy_lik,
                        const __nv_bfloat16* __restrict__ d_dec, const __nv_bfloat16* __restrict__ d_ctx,
                        const __nv_bfloat16* __restrict__ d_abs, long total, __nv_bfloat16* __restrict__ dy) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  float g = dy_lik ? dy_lik[i] : 0.0f;
  if (d_dec) g += __bfloat162float(d_dec[i]);
  if (d_ctx) g += __bfloat162float(d_ctx[i]);
  if (d_abs) {
    const float v = y[i];
    const float s = v > 0.0f ? 1.0f : (v < 0.0f ? -1.0f : 0.0f);
    g += s * __bfloat162float(d_abs[i]);
  }
  dy[i] = __float2bfloat16_rn(g);
}

// out(bf16) = a(fp32) + b(bf16)
__global__ void __launch_bounds__(256)
add_f32_bf16_kernel(const float* __restrict__ a, const __nv_bfloat16* __restrict__ b, long total,
                    __nv_bfloat16* __restrict__ out) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  out[i] = __float2bfloat16_rn(a[i] + __bfloat162float(b[i]));
}

// fused[p] = cat(P2[p] * w0, C2[p] * w1, (y1w[p] + noise[p]) * w2)      MASIC.py:827 (training)
// one warp per pixel
__global__ void __launch_bounds__(256)
mask_fuse_fwd_kernel(const __nv_bfloat16* __restrict__ P2, const __nv_bfloat16* __restrict__ C2, int c2,
                     const float* __restrict__ y1w, const float* __restrict__ noise, int m,
                     const float* __restrict__ mw, long npix, __nv_bfloat16* __restrict__ fused) {
  const long p = blockIdx.x * 8L + (threadIdx.x >> 5);
  if (p >= npix) return;
  const int lane = threadIdx.x & 31;
  const float w0 = mw[p * 3], w1 = mw[p * 3 + 1], w2 = mw[p * 3 + 2];
  const int pitch = 2 * c2 + m;
  __nv_bfloat16* o = fused + p * pitch;
  for (int c = lane * 2; c < c2; c += 64) {
    const float2 a = ld_bf2(P2 + p * c2 + c), b = ld_bf2(C2 + p * c2 + c);
    st_bf2(o + c, a.x * w0, a.y * w0);
    st_bf2(o + c2 + c, b.x * w1, b.y * w1);
  }
  for (int c = lane; c < m; c += 32) o[2 * c2 + c] = __float2bfloat16_rn((y1w[p * m + c] + noise[p * m + c]) * w2);
}

// backward of the above: dP2 = g[0:c2] w0, dC2 = g[c2:2c2] w1, dY = g[2c2:] w2,  dmw[j] = sum_c g * value
__global__ void __launch_bounds__(256)
mask_fuse_bwd_kernel(const __nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ P2,
                     const __nv_bfloat16* __restrict__ C2, int c2, const float* __restrict__ y1w,
                     const float* __restrict__ noise, int m, const float* __restrict__ mw, long npix,
                     __nv_bfloat16* __restrict__ dP2, __nv_bfloat16* __restrict__ dC2, __nv_bfloat16* __restrict__ dY,
                     float* __restrict__ dmw) {
  const long p = blockIdx.x * 8L + (threadIdx.x >> 5);
  if (p >= npix) return;
  const int lane = threadIdx.x & 31;
  const float w0 = mw[p * 3], w1 = mw[p * 3 + 1], w2 = mw[p * 3 + 2];
  const int pitch = 2 * c2 + m;
  const __nv_bfloat16* gp = g + p * pitch;
  float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
  for (int c = lane * 2; c < c2; c += 64) {
    const float2 ga = ld_bf2(gp + c), gb = ld_bf2(gp + c2 + c);
    const float2 a = ld_bf2(P2 + p * c2 + c), b = ld_bf2(C2 + p * c2 + c);
    s0 += ga.x * a.x + ga.y * a.y;
    s1 += gb.x * b.x + gb.y * b.y;
    st_bf2(dP2 + p * c2 + c, ga.x * w0, ga.y * w0);
    st_bf2(dC2 + p * c2 + c, gb.x * w1, gb.y * w1);
  }
  for (int c = lane; c < m; c += 32) {
    const float gv = __bfloat162float(gp[2 * c2 + c]);
    s2 += gv * (y1w[p * m + c] + noise[p * m + c]);
    dY[p * m + c] = __float2bfloat16_rn(gv * w2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if (lane == 0) { dmw[p * 3] = s0; dmw[p * 3 + 1] = s1; dmw[p * 3 + 2] = s2; }
}

inline dim3 cs_grid(long npix, int C) { return dim3((C + 63) / 64, (unsigned)((npix + PIX_PER_BLOCK - 1) / PIX_PER_BLOCK)); }

}  // namespace

#define S(stream) static_cast<cudaStream_t>(stream)
#define BF(p) static_cast<__nv_bfloat16*>(p)
#define CBF(p) static_cast<const __nv_bfloat16*>(p)

extern "C" int masic_act_bwd_bias(void* g_bf16, int g_pitch, int g_coff, const void* y_bf16, int y_pitch, int y_coff,
                                  int act, int64_t n_pixels, int c, float* bias_grad, void* stream) {
  if (!g_bf16 || n_pixels <= 0 || c <= 0 || (c & 1) || (g_pitch & 1) || (g_coff & 1)) return MASIC_EINVAL;
  if (act != MASIC_ACT_NONE && (!y_bf16 || (y_pitch & 1) || (y_coff & 1))) return MASIC_EINVAL;
  if (act == MASIC_ACT_NONE && !bias_grad) return MASIC_OK;
  if (act == MASIC_ACT_NONE)
    colsum_bf16_kernel<<<cs_grid(n_pixels, c), dim3(32, 8), 0, S(stream)>>>(CBF(g_bf16), g_pitch, g_coff, n_pixels, c,
                                                                             bias_grad);
  else
    act_bwd_bias_kernel<<<cs_grid(n_pixels, c), dim3(32, 8), 0, S(stream)>>>(BF(g_bf16), g_pitch, g_coff, CBF(y_bf16),
                                                                              y_pitch, y_coff, act, n_pixels, c, bias_grad);
  return (int)cudaGetLastError();
}

extern "C" int masic_act_bwd_bias_out(const void* g_bf16, int g_pitch, int g_coff, const void* y_bf16, int y_pitch,
                                      int y_coff, int act, int64_t n_pixels, int c, void* dst_bf16, int dst_pitch,
                                      int dst_coff, float* bias_grad, void* stream) {
  if (!g_bf16 || !dst_bf16 || n_pixels <= 0 || c <= 0 || (c & 1) || (g_pitch & 1) || (g_coff & 1) || (dst_pitch & 1) ||
      (dst_coff & 1) || dst_coff + c > dst_pitch || g_coff + c > g_pitch)
    return MASIC_EINVAL;
  if (act != MASIC_ACT_NONE && (!y_bf16 || (y_pitch & 1) || (y_coff & 1) || y_coff + c > y_pitch)) return MASIC_EINVAL;
  act_bwd_bias_out_kernel<<<cs_grid(n_pixels, c), dim3(32, 8), 0, S(stream)>>>(
      CBF(g_bf16), g_pitch, g_coff, CBF(y_bf16), y_pitch, y_coff, act, n_pixels, c, BF(dst_bf16), dst_pitch, dst_coff,
      bias_grad);
  return (int)cudaGetLastError();
}

extern "C" int masic_gdn_square(const void* x_bf16, void* sq_bf16, int64_t numel, void* stream) {
  if (!x_bf16 || !sq_bf16 || numel <= 0 || (numel & 1)) return MASIC_EINVAL;
  gdn_sq_kernel<<<(unsigned)((numel / 2 + 255) / 256), 256, 0, S(stream)>>>(CBF(x_bf16), BF(sq_bf16), numel / 2);
  return (int)cudaGetLastError();
}

extern "C" int masic_gdn_apply(const void* x_bf16, const float* norm, int inverse, void* y_bf16, int64_t numel,
                               void* stream) {
  if (!x_bf16 || !norm || !y_bf16 || numel <= 0 || (numel & 1)) return MASIC_EINVAL;
  gdn_apply_kernel<<<(unsigned)((numel / 2 + 255) / 256), 256, 0, S(stream)>>>(CBF(x_bf16), norm, inverse, BF(y_bf16),
                                                                               numel / 2);
  return (int)cudaGetLastError();
}

extern "C" int masic_gdn_bwd_a(void* g_bf16, const void* x_bf16, const float* norm, int inverse, void* t_bf16,
                               int64_t n_pixels, int c, float* dbeta_prime, void* stream) {
  if (!g_bf16 || !x_bf16 || !norm || !t_bf16 || n_pixels <= 0 || c <= 0 || (c & 1)) return MASIC_EINVAL;
  gdn_bwd_a_kernel<<<cs_grid(n_pixels, c), dim3(32, 8), 0, S(stream)>>>(BF(g_bf16), CBF(x_bf16), norm, inverse,
                                                                         BF(t_bf16), n_pixels, c, dbeta_prime);
  return (int)cudaGetLastError();
}

extern "C" int masic_gdn_bwd_b(void* u_bf16, const void* x_bf16, const float* v, int64_t n_pixels, int c,
                               float* dbias, void* stream) {
  if (!u_bf16 || !x_bf16 || !v || n_pixels <= 0 || c <= 0 || (c & 1)) return MASIC_EINVAL;
  gdn_bwd_b_kernel<<<cs_grid(n_pixels, c), dim3(32, 8), 0, S(stream)>>>(BF(u_bf16), CBF(x_bf16), v, n_pixels, c, dbias);
  return (int)cudaGetLastError();
}

extern "C" int masic_reparam_bwd(const float* dprime, const float* stored, int n, float minimum, int accumulate,
                                 float* dstored, void* stream) {
  if (!dprime || !stored || !dstored || n <= 0) return MASIC_EINVAL;
  const float bound = sqrtf(minimum + 1.4551915228366852e-11f);
  reparam_bwd_kernel<<<(n + 255) / 256, 256, 0, S(stream)>>>(dprime, stored, n, bound, accumulate, dstored);
  return (int)cudaGetLastError();
}

struct MasicReparamBatch { ReparamJob* d_jobs; int n_jobs; int max_n; };

extern "C" int masic_reparam_batch_create(const float* const* dprime, const float* const* stored, float* const* dstored,
                                          const int* numel, const float* minimum, const int* accumulate, int n_jobs,
                                          MasicReparamBatch** out) {
  if (!dprime || !stored || !dstored || !numel || !minimum || !out || n_jobs <= 0 || n_jobs > 4096) return MASIC_EINVAL;
  ReparamJob* h = new ReparamJob[n_jobs];
  int max_n = 0;
  for (int i = 0; i < n_jobs; ++i) {
    if (!dprime[i] || !stored[i] || !dstored[i] || numel[i] <= 0) { delete[] h; return MASIC_EINVAL; }
    h[i].dprime = dprime[i]; h[i].stored = stored[i]; h[i].dstored = dstored[i]; h[i].n = numel[i];
    h[i].bound = sqrtf(minimum[i] + 1.4551915228366852e-11f);
    h[i].accumulate = accumulate ? accumulate[i] : 0; h[i].pad = 0;
    if (numel[i] > max_n) max_n = numel[i];
  }
  MasicReparamBatch* b = new MasicReparamBatch();
  b->n_jobs = n_jobs; b->max_n = max_n; b->d_jobs = nullptr;
  cudaError_t e = cudaMalloc(&b->d_jobs, sizeof(ReparamJob) * n_jobs);
  if (e == cudaSuccess) e = cudaMemcpy(b->d_jobs, h, sizeof(ReparamJob) * n_jobs, cudaMemcpyHostToDevice);
  delete[] h;
  if (e != cudaSuccess) { if (b->d_jobs) cudaFree(b->d_jobs); delete b; return (int)e; }
  *out = b;
  return MASIC_OK;
}

extern "C" int masic_reparam_batch_launch(const MasicReparamBatch* b, void* stream) {
  if (!b) return MASIC_EINVAL;
  int gx = (b->max_n + 255) / 256;
  if (gx > 64) gx = 64;
  reparam_bwd_batch_kernel<<<dim3(gx, b->n_jobs), 256, 0, S(stream)>>>(b->d_jobs);
  return (int)cudaGetLastError();
}

extern "C" void masic_reparam_batch_destroy(MasicReparamBatch* b) {
  if (!b) return;
  if (b->d_jobs) cudaFree(b->d_jobs);
  delete b;
}

extern "C" int masic_latent_prep_train(const float* y_nhwc, const float* noise_nhwc, int64_t n_pixels, int c,
                                       void* y_abs_bf16, int abs_pitch, void* y_noisy_bf16, int noisy_pitch,
                                       void* stream) {
  if (!y_nhwc || n_pixels <= 0 || c <= 0 || (y_noisy_bf16 && !noise_nhwc)) return MASIC_EINVAL;
  const long total = (long)n_pixels * c;
  latent_prep_train_kernel<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(
      y_nhwc, noise_nhwc, total, c, BF(y_abs_bf16), abs_pitch, BF(y_noisy_bf16), noisy_pitch);
  return (int)cudaGetLastError();
}

extern "C" int masic_latent_merge_bwd(const float* y_nhwc, const float* dy_lik, const void* d_dec_bf16,
                                      const void* d_ctx_bf16, const void* d_abs_bf16, int64_t numel, void* dy_bf16,
                                      void* stream) {
  if (!dy_bf16 || numel <= 0 || (d_abs_bf16 && !y_nhwc)) return MASIC_EINVAL;
  latent_merge_bwd_kernel<<<(unsigned)((numel + 255) / 256), 256, 0, S(stream)>>>(
      y_nhwc, dy_lik, CBF(d_dec_bf16), CBF(d_ctx_bf16), CBF(d_abs_bf16), numel, BF(dy_bf16));
  return (int)cudaGetLastError();
}

extern "C" int masic_add_f32_bf16(const float* a, const void* b_bf16, int64_t numel, void* out_bf16, void* stream) {
  if (!a || !b_bf16 || !out_bf16 || numel <= 0) return MASIC_EINVAL;
  add_f32_bf16_kernel<<<(unsigned)((numel + 255) / 256), 256, 0, S(stream)>>>(a, CBF(b_bf16), numel, BF(out_bf16));
  return (int)cudaGetLastError();
}

extern "C" int masic_mask_fuse_fwd(const void* p2_bf16, const void* c2_bf16, int c2, const float* y1w_nhwc,
                                   const float* noise_nhwc, int m, const float* mask_weights_nhwc, int64_t n_pixels,
                                   void* fused_bf16, void* stream) {
  if (!p2_bf16 || !c2_bf16 || !y1w_nhwc || !noise_nhwc || !mask_weights_nhwc || !fused_bf16 || (c2 & 1) || n_pixels <= 0)
    return MASIC_EINVAL;
  mask_fuse_fwd_kernel<<<(unsigned)((n_pixels + 7) / 8), 256, 0, S(stream)>>>(
      CBF(p2_bf16), CBF(c2_bf16), c2, y1w_nhwc, noise_nhwc, m, mask_weights_nhwc, n_pixels, BF(fused_bf16));
  return (int)cudaGetLastError();
}

extern "C" int masic_mask_fuse_bwd(const void* g_bf16, const void* p2_bf16, const void* c2_bf16, int c2,
                                   const float* y1w_nhwc, const float* noise_nhwc, int m,
                                   const float* mask_weights_nhwc, int64_t n_pixels, void* dp2_bf16, void* dc2_bf16,
                                   void* dy1w_bf16, float* dmask_weights_nhwc, void* stream) {
  if (!g_bf16 || !p2_bf16 || !c2_bf16 || !y1w_nhwc || !noise_nhwc || !mask_weights_nhwc || !dp2_bf16 || !dc2_bf16 ||
      !dy1w_bf16 || !dmask_weights_nhwc || (c2 & 1) || n_pixels <= 0)
    return MASIC_EINVAL;
  mask_fuse_bwd_kernel<<<(unsigned)((n_pixels + 7) / 8), 256, 0, S(stream)>>>(
      CBF(g_bf16), CBF(p2_bf16), CBF(c2_bf16), c2, y1w_nhwc, noise_nhwc, m, mask_weights_nhwc, n_pixels, BF(dp2_bf16),
      BF(dc2_bf16), BF(dy1w_bf16), dmask_weights_nhwc);
  return (int)cudaGetLastError();
}
