// entropy.cu — fused, memory-bound entropy-model kernels (sm_100a).
//
// Replaces (reference, file:line):
//   GaussianMixtureConditional_gf.forward/_likelihood  compressai/entropy_models/entropy_models.py:808-858
//   (+ the softmax over K of MASIC.py:389-393 / :459-464 when the weights arrive as logits)
//   EntropyBottleneck.forward/_likelihood/_logits_cumulative        entropy_models.py:350-411
//   GaussianConditional._likelihood/forward/build_indexes           entropy_models.py:528-562
//   EntropyModel._quantize('symbols'|'dequantize')                  entropy_models.py:98-125
//
// Layout: every tensor argument is described by (stride_n, stride_c, stride_p) in elements,
// p = y*W + x, so the same kernel serves the reference's NCHW tensors (stride_c = H*W,
// stride_p = 1) and the engine's NHWC buffers (stride_c = 1, stride_p = C).  Blocks walk
// 32 channels x 32 positions through a shared-memory transpose so that both sides of a
// layout change stay coalesced.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"

namespace {

constexpr float kLikBound = 1e-9f;
constexpr float kInvSqrt2Neg = -0.70710678118654752440f;   // float(-(2**-0.5))

// erfc with fractional error < 1.2e-7 (+ fp32 evaluation error) everywhere, branch-free: the Chebyshev fit of
// Numerical Recipes' erfcc(), erfc(|x|) = t * exp(-x^2 + P(t)), t = 2 / (2 + |x|).  CUDA's erfcf() costs ~160 issued
// instructions per call on this data (its argument regimes diverge inside every warp), which made the mixture
// likelihood kernel ALU-bound at 28 % of HBM peak; this one is ~30.
__device__ __forceinline__ float erfc_fit(float x) {
  const float z = fabsf(x);
  const float t = __fdividef(2.0f, 2.0f + z);      // MUFU.RCP + FMUL; an IEEE division is ~50 issued instructions
  float p = 0.17087277f;
  p = fmaf(p, t, -0.82215223f);
  p = fmaf(p, t, 1.48851587f);
  p = fmaf(p, t, -1.13520398f);
  p = fmaf(p, t, 0.27886807f);
  p = fmaf(p, t, -0.18628806f);
  p = fmaf(p, t, 0.09678418f);
  p = fmaf(p, t, 0.37409196f);
  p = fmaf(p, t, 1.00002368f);
  p = fmaf(p, t, -1.26551223f);
  const float r = t * __expf(fmaf(-z, z, p));       // ex2.approx: 2 ulp + |arg| * 2^-23 relative, far inside the tolerance
  return x >= 0.0f ? r : 2.0f - r;
}

__device__ __forceinline__ float phi_exact(float x) { return 0.5f * erfcf(kInvSqrt2Neg * x); }
#ifdef MASIC_EXACT_ERFC
__device__ __forceinline__ float phi(float x) { return phi_exact(x); }
#else
__device__ __forceinline__ float phi(float x) { return 0.5f * erfc_fit(kInvSqrt2Neg * x); }
#endif

#ifdef MASIC_EXACT_ERFC
__device__ __forceinline__ float gauss_mass(float v_abs, float s) {
  return phi((0.5f - v_abs) / s) - phi((-0.5f - v_abs) / s);
}
#else
// one approximate reciprocal (<= 1 ulp) instead of two IEEE divisions: the argument of erfc moves by <= 2 ulp
__device__ __forceinline__ float gauss_mass(float v_abs, float s) {
  const float inv_s = __fdividef(1.0f, s);
  return phi((0.5f - v_abs) * inv_s) - phi((-0.5f - v_abs) * inv_s);
}
#endif

struct View { long sn, sc, sp; };
__device__ __forceinline__ long at(const View& v, int n, int c, int p) {
  return n * v.sn + c * v.sc + (long)p * v.sp;
}

// ------------------------------------------------------------------ K-component mixture
// grid: (ceil(P/32), ceil(M/32), N); block (32, 8).
// `fast_c` != 0: parameters are channel-fastest (NHWC): threadIdx.x walks channels while loading.
template <int K>
__global__ void __launch_bounds__(256)
gmm_fwd_kernel(const float* __restrict__ y, View vy, const float* __restrict__ sigma,
               const float* __restrict__ mu, const float* __restrict__ wgt, View vp, int w_is_logits,
               int fast_c, int M, int P, float scale_bound, float* __restrict__ y_hat,
               float* __restrict__ lik, View vo, int32_t* __restrict__ sym,
               __nv_bfloat16* __restrict__ yq_bf16, int bf_pitch, int bf_coff, int f16,
               const float* __restrict__ rowscale, int rs_stride, int rs_off) {
  __shared__ float s_lik[32][33];
  __shared__ float s_yh[32][33];
  const int n = blockIdx.z;
  const int p0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  // ---- compute phase: pick the mapping that makes the 3K parameter loads coalesced.  Each thread walks four
  // (position, channel) elements; the 16 loads of the NEXT element are issued before the current one is evaluated
  // (the kernel was bound by the latency of loads consumed right where they were issued).
  struct Elem { float y, s[K], m[K], w[K]; bool ok; int pl, ml; };
  auto fetch = [&](int j) {
    Elem e;
    e.pl = fast_c ? j : threadIdx.x;
    e.ml = fast_c ? threadIdx.x : j;
    const int p = p0 + e.pl, m = m0 + e.ml;
    e.ok = j < 32 && p < P && m < M;
    e.y = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) { e.s[k] = 1.0f; e.m[k] = 0.0f; e.w[k] = 0.0f; }
    if (e.ok) {
      e.y = __ldg(y + at(vy, n, m, p));
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const long o = at(vp, n, k * M + m, p);
        e.s[k] = __ldg(sigma + o); e.m[k] = __ldg(mu + o); e.w[k] = __ldg(wgt + o);
      }
    }
    return e;
  };
  Elem cur = fetch(threadIdx.y);
  for (int j = threadIdx.y; j < 32; j += 8) {
    const Elem nxt = fetch(j + 8);
    float l = 0.0f, yh = 0.0f;
    if (cur.ok) {
      yh = rintf(cur.y);
      float wk[K];
      if (w_is_logits) {
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < K; ++k) { wk[k] = cur.w[k]; mx = fmaxf(mx, wk[k]); }
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < K; ++k) { wk[k] = expf(wk[k] - mx); sum += wk[k]; }
        const float inv_sum = 1.0f / sum;                    // one IEEE division instead of K
#pragma unroll
        for (int k = 0; k < K; ++k) wk[k] *= inv_sum;
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) wk[k] = cur.w[k];
      }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float s = fmaxf(cur.s[k], scale_bound);
        const float v = fabsf(yh - cur.m[k]);
        l += gauss_mass(v, s) * wk[k];
      }
      l = fmaxf(l, kLikBound);
    }
    s_lik[cur.pl][cur.ml] = l;
    s_yh[cur.pl][cur.ml] = yh;
    cur = nxt;
  }
  __syncthreads();
  // ---- store phase: fastest output dimension on threadIdx.x
  const bool out_fast_c = vo.sc == 1;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int pl = out_fast_c ? j : threadIdx.x;
    const int ml = out_fast_c ? threadIdx.x : j;
    const int p = p0 + pl, m = m0 + ml;
    if (p < P && m < M) {
      const long o = at(vo, n, m, p);
      if (lik) lik[o] = s_lik[pl][ml];
      if (y_hat) y_hat[o] = s_yh[pl][ml];
      if (sym) sym[o] = (int32_t)s_yh[pl][ml];
    }
  }
  if (yq_bf16) {   // NHWC bf16 copy of round(y) for the next conv (optionally mask-weighted)
    for (int j = threadIdx.y; j < 32; j += 8) {
      const int p = p0 + j, m = m0 + threadIdx.x;
      if (p < P && m < M) {
        float v = s_yh[j][threadIdx.x];
        if (rowscale) v *= rowscale[((long)n * P + p) * rs_stride + rs_off];
        reinterpret_cast<uint16_t*>(yq_bf16)[((long)n * P + p) * bf_pitch + bf_coff + m] = masic::pack16(v, f16);
      }
    }
  }
}

// The engine's configuration (parameters NHWC, weight logits, outputs NCHW) with 128-bit loads: a thread owns FOUR
// consecutive channels of one position, so its 16 parameter loads are LDG.128 (4x fewer load instructions than the
// generic kernel, all independent and in flight together) and a warp touches 4 positions x 128 contiguous bytes per
// load.  Results go through a 32 x 32 shared-memory transpose so the NCHW stores are coalesced along positions.
// Same per-element arithmetic as gmm_fwd_kernel: bit-identical outputs.  block (8, 32): x = channel quad, y = position.
template <int K>
__global__ void __launch_bounds__(256)
gmm_fwd_nhwc_v4_kernel(const float* __restrict__ y, const float* __restrict__ sigma, const float* __restrict__ mu,
                       const float* __restrict__ wgt, int M, int P, float scale_bound, float* __restrict__ y_hat,
                       float* __restrict__ lik) {
  __shared__ float s_lik[32][33];
  __shared__ float s_yh[32][33];
  const int n = blockIdx.z;
  const int p0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  const int p = p0 + threadIdx.y, m = m0 + 4 * threadIdx.x;
  if (p < P && m < M) {
    const size_t row = (static_cast<size_t>(n) * P + p);
    const float4 yv = __ldg(reinterpret_cast<const float4*>(y + row * M + m));
    float4 sv[K], mv[K], wv[K];
    const size_t pb = row * (static_cast<size_t>(K) * M) + m;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      sv[k] = __ldg(reinterpret_cast<const float4*>(sigma + pb + static_cast<size_t>(k) * M));
      mv[k] = __ldg(reinterpret_cast<const float4*>(mu + pb + static_cast<size_t>(k) * M));
      wv[k] = __ldg(reinterpret_cast<const float4*>(wgt + pb + static_cast<size_t>(k) * M));
    }
    const float ye[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float wk[K], sk[K], mk[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float* sp = reinterpret_cast<const float*>(&sv[k]);
        const float* mp = reinterpret_cast<const float*>(&mv[k]);
        const float* wp = reinterpret_cast<const float*>(&wv[k]);
        sk[k] = sp[e]; mk[k] = mp[e]; wk[k] = wp[e];
      }
      const float yh = rintf(ye[e]);
      float mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < K; ++k) mx = fmaxf(mx, wk[k]);
      float sum = 0.0f;
#pragma unroll
      for (int k = 0; k < K; ++k) { wk[k] = expf(wk[k] - mx); sum += wk[k]; }
      const float inv_sum = 1.0f / sum;
#pragma unroll
      for (int k = 0; k < K; ++k) wk[k] *= inv_sum;
      float l = 0.0f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float sd = fmaxf(sk[k], scale_bound);
        const float v = fabsf(yh - mk[k]);
        l += gauss_mass(v, sd) * wk[k];
      }
      s_lik[threadIdx.y][4 * threadIdx.x + e] = fmaxf(l, kLikBound);
      s_yh[threadIdx.y][4 * threadIdx.x + e] = yh;
    }
  }
  __syncthreads();
  // store: thread (tx, ty) -> flat id; position fastest
  const int tid = threadIdx.y * 8 + threadIdx.x;
  const int pl = tid & 31;
  for (int ml = tid >> 5; ml < 32; ml += 8) {
    const int pp = p0 + pl, mm = m0 + ml;
    if (pp < P && mm < M) {
      const size_t o = (static_cast<size_t>(n) * M + mm) * P + pp;
      lik[o] = s_lik[pl][ml];
      y_hat[o] = s_yh[pl][ml];
    }
  }
}

// ------------------------------------------------------------------ single Gaussian
__global__ void __launch_bounds__(256)
gc_fwd_kernel(const float* __restrict__ y, const float* __restrict__ scales,
              const float* __restrict__ means, long total, float scale_bound,
              float* __restrict__ y_hat, float* __restrict__ lik, int32_t* __restrict__ sym) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float mu = means ? means[i] : 0.0f;
  float r = y[i];
  if (means) r = r - mu;
  r = rintf(r);
  if (sym) sym[i] = (int32_t)r;
  const float deq = means ? r + mu : r;
  if (y_hat) y_hat[i] = deq;
  if (lik) {
    const float v = means ? fabsf(deq - mu) : fabsf(deq);
    const float s = fmaxf(scales[i], scale_bound);
    lik[i] = fmaxf(gauss_mass(v, s), kLikBound);
  }
}

// idx = (L-1) - #{ j < L-1 : max(scale, bound) <= table[j] }   (table ascending)
__global__ void __launch_bounds__(256)
gc_indexes_kernel(const float* __restrict__ scales, long total, const float* __restrict__ table, int L,
                  float scale_bound, int32_t* __restrict__ idx) {
  extern __shared__ float s_tab[];
  for (int j = threadIdx.x; j < L; j += blockDim.x) s_tab[j] = table[j];
  __syncthreads();
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float s = fmaxf(scales[i], scale_bound);
  // first j in [0, L-1) with table[j] >= s ; count of (s <= table[j]) = (L-1) - j
  int lo = 0, hi = L - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (s_tab[mid] >= s) hi = mid; else lo = mid + 1;
  }
  idx[i] = lo;      // (L-1) - ((L-1) - lo)
}

// ------------------------------------------------------------------ EntropyBottleneck
// per-channel parameter block prepared once per launch: softplus(matrices), biases, tanh(factors)
struct EBChan {
  float m0[3], m1[9], m2[9], m3[9], m4[3];
  float b0[3], b1[3], b2[3], b3[3], b4[1];
  float f0[3], f1[3], f2[3], f3[3];
  float median;
};

__device__ __forceinline__ float softplus_f(float x) { return x > 20.0f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ float eb_logits(const EBChan& c, float v) {
  float a[3], t[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    a[i] = c.m0[i] * v + c.b0[i];
    a[i] += c.f0[i] * tanhf(a[i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    t[i] = c.m1[i * 3] * a[0] + c.m1[i * 3 + 1] * a[1] + c.m1[i * 3 + 2] * a[2] + c.b1[i];
    t[i] += c.f1[i] * tanhf(t[i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    a[i] = c.m2[i * 3] * t[0] + c.m2[i * 3 + 1] * t[1] + c.m2[i * 3 + 2] * t[2] + c.b2[i];
    a[i] += c.f2[i] * tanhf(a[i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    t[i] = c.m3[i * 3] * a[0] + c.m3[i * 3 + 1] * a[1] + c.m3[i * 3 + 2] * a[2] + c.b3[i];
    t[i] += c.f3[i] * tanhf(t[i]);
  }
  return c.m4[0] * t[0] + c.m4[1] * t[1] + c.m4[2] * t[2] + c.b4[0];
}

// grid (ceil(P/256), C, N)
__global__ void __launch_bounds__(256)
eb_fwd_kernel(const float* __restrict__ z, View vz, int P,
              const float* __restrict__ mat0, const float* __restrict__ mat1,
              const float* __restrict__ mat2, const float* __restrict__ mat3,
              const float* __restrict__ mat4, const float* __restrict__ b0,
              const float* __restrict__ b1, const float* __restrict__ b2,
              const float* __restrict__ b3, const float* __restrict__ b4,
              const float* __restrict__ f0, const float* __restrict__ f1,
              const float* __restrict__ f2, const float* __restrict__ f3,
              const float* __restrict__ quantiles, float* __restrict__ z_hat,
              float* __restrict__ lik, View vo, int32_t* __restrict__ sym,
              __nv_bfloat16* __restrict__ zq_bf16, int bf_pitch, int f16) {
  __shared__ EBChan sc;
  const int c = blockIdx.y, n = blockIdx.z;
  if (threadIdx.x < 3) {
    const int i = threadIdx.x;
    sc.m0[i] = softplus_f(mat0[c * 3 + i]);  sc.m4[i] = softplus_f(mat4[c * 3 + i]);
    sc.b0[i] = b0[c * 3 + i]; sc.b1[i] = b1[c * 3 + i]; sc.b2[i] = b2[c * 3 + i]; sc.b3[i] = b3[c * 3 + i];
    sc.f0[i] = tanhf(f0[c * 3 + i]); sc.f1[i] = tanhf(f1[c * 3 + i]);
    sc.f2[i] = tanhf(f2[c * 3 + i]); sc.f3[i] = tanhf(f3[c * 3 + i]);
  }
  if (threadIdx.x < 9) {
    const int i = threadIdx.x;
    sc.m1[i] = softplus_f(mat1[c * 9 + i]); sc.m2[i] = softplus_f(mat2[c * 9 + i]);
    sc.m3[i] = softplus_f(mat3[c * 9 + i]);
  }
  if (threadIdx.x == 0) { sc.b4[0] = b4[c]; sc.median = quantiles[c * 3 + 1]; }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const float med = sc.median;
  const float r = rintf(z[at(vz, n, c, p)] - med);
  const float q = r + med;
  const long o = at(vo, n, c, p);
  if (sym) sym[o] = (int32_t)r;
  if (z_hat) z_hat[o] = q;
  if (zq_bf16) reinterpret_cast<uint16_t*>(zq_bf16)[((long)n * P + p) * bf_pitch + c] = masic::pack16(q, f16);
  if (lik) {
    const float lower = eb_logits(sc, q - 0.5f);
    const float upper = eb_logits(sc, q + 0.5f);
    const float su = lower + upper;
    const float sign = su > 0.0f ? -1.0f : (su < 0.0f ? 1.0f : 0.0f);
    lik[o] = fmaxf(fabsf(sigmoid_f(sign * upper) - sigmoid_f(sign * lower)), kLikBound);
  }
}

__global__ void __launch_bounds__(256)
quantize_kernel(const float* __restrict__ x, const float* __restrict__ means, long total,
                float* __restrict__ deq, int32_t* __restrict__ sym) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  float r = x[i];
  const float mu = means ? means[i] : 0.0f;
  if (means) r = r - mu;
  r = rintf(r);
  if (sym) sym[i] = (int32_t)r;
  if (deq) deq[i] = means ? r + mu : r;
}

// |y| and round(y) as bf16 NHWC copies of an fp32 NHWC latent (inputs of h_a, context conv, decoder)
__global__ void __launch_bounds__(256)
latent_prep_kernel(const float* __restrict__ y, long total, int C, __nv_bfloat16* __restrict__ y_abs,
                   int abs_pitch, __nv_bfloat16* __restrict__ y_round, int rnd_pitch, int rnd_coff,
                   const float* __restrict__ rowscale, int rs_stride, int rs_off, int f16) {
  // four channels per thread when the layout allows (16-byte loads, 8-byte stores), else one
  const bool v4 = (C & 3) == 0 && (abs_pitch & 3) == 0 && (rnd_pitch & 3) == 0 && (rnd_coff & 3) == 0;
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (v4) {
    const unsigned c4 = (unsigned)C >> 2;
    if (i >= (total >> 2)) return;
    const unsigned pix = (unsigned)(i / c4);           // total / 4 < 2^32 for every tensor this runs on
    const int c = (int)((unsigned)i - pix * c4) * 4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(y) + i);
    if (y_abs) {
      *reinterpret_cast<uint2*>(y_abs + (long)pix * abs_pitch + c) =
          make_uint2(masic::pack16x2(fabsf(v.x), fabsf(v.y), f16), masic::pack16x2(fabsf(v.z), fabsf(v.w), f16));
    }
    if (y_round) {
      const float s = rowscale ? rowscale[(long)pix * rs_stride + rs_off] : 1.0f;
      float r0 = rintf(v.x), r1 = rintf(v.y), r2 = rintf(v.z), r3 = rintf(v.w);
      if (rowscale) { r0 *= s; r1 *= s; r2 *= s; r3 *= s; }
      *reinterpret_cast<uint2*>(y_round + (long)pix * rnd_pitch + rnd_coff + c) =
          make_uint2(masic::pack16x2(r0, r1, f16), masic::pack16x2(r2, r3, f16));
    }
    return;
  }
  if (i >= total) return;
  const long pix = i / C;
  const int c = (int)(i - pix * C);
  const float v = y[i];
  if (y_abs) reinterpret_cast<uint16_t*>(y_abs)[pix * abs_pitch + c] = masic::pack16(fabsf(v), f16);
  if (y_round) {
    float r = rintf(v);
    if (rowscale) r *= rowscale[pix * rs_stride + rs_off];
    reinterpret_cast<uint16_t*>(y_round)[pix * rnd_pitch + rnd_coff + c] = masic::pack16(r, f16);
  }
}


// ------------------------------------------------------------------ per-symbol CDFs of the y bitstream
// HSIC.compress / decompress (MASIC.py:1006-1043, :1263-1300): for latent element (p, ch) the coder model is
//   pmf[s]  = sum_k w_k [Phi((.5 - |s - (mu_k + minmax)|)/max(sigma_k, bound)) - Phi((-.5 - |..|)/..)],  s = 0..2*minmax
//   pmf     = round(clip(pmf, 1/65536, 1) / sum(clip) * 65536)          (float32 throughout)
//   cdf     = [0] + cumsum(pmf)                                         (its total need not be 65536)
// One warp per (position, listed channel).  rows != NULL writes the whole row (L+1 int32, L = 2*minmax+1), which
// the decoder searches; intervals != NULL writes (cdf[sym], cdf[sym+1]-cdf[sym], cdf[L]) for the known symbol
// sym = y_hat + minmax — all an encoder needs.
//
// EXACTNESS.  The reference evaluates the pmf with separate torch ops on cuda:0 (MASIC.py:988-1022: sub, abs, div,
// mul, erfc, mul, sub, mul, add — each an IEEE fp32 kernel) and the normalisation with NumPy on the host
// (:1040-1043, float32: np.clip, np.sum, /, *, np.round, np.add.accumulate).  Every operation below is therefore a
// single correctly rounded fp32 operation in the same order (the _rn intrinsics keep nvcc from contracting them into
// FMAs), erfc is CUDA's erfcf (what torch calls), and the sum of the clipped pmf follows NumPy's pairwise summation
// order (blocks of <= 128 with eight interleaved accumulators, halves split at multiples of 8), so that the integer
// rows are IDENTICAL to the reference's, not just close (tests/test_bitstream_gpu.py).

// np.sum over a contiguous float32 vector (numpy/_core/src/umath/loops_utils.h.src, *_pairwise_sum): all lanes
// call this with the same arguments and get the same result.
__device__ float numpy_pairwise_sum(const float* a, int n, int lane) {
  if (n < 8) {
    float r = -0.0f;
    for (int i = 0; i < n; ++i) r = __fadd_rn(r, a[i]);
    return r;
  }
  if (n <= 128) {
    const int j = lane & 7;                       // lane j (and its copies j+8, j+16, j+24) owns accumulator j
    float r = a[j];
    const int body = n - (n & 7);
    for (int i = 8; i < body; i += 8) r = __fadd_rn(r, a[i + j]);
    const float r0 = __shfl_sync(0xffffffffu, r, 0), r1 = __shfl_sync(0xffffffffu, r, 1);
    const float r2 = __shfl_sync(0xffffffffu, r, 2), r3 = __shfl_sync(0xffffffffu, r, 3);
    const float r4 = __shfl_sync(0xffffffffu, r, 4), r5 = __shfl_sync(0xffffffffu, r, 5);
    const float r6 = __shfl_sync(0xffffffffu, r, 6), r7 = __shfl_sync(0xffffffffu, r, 7);
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r0, r1), __fadd_rn(r2, r3)),
                          __fadd_rn(__fadd_rn(r4, r5), __fadd_rn(r6, r7)));
    for (int i = body; i < n; ++i) res = __fadd_rn(res, a[i]);
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 & 7;
  const float lo = numpy_pairwise_sum(a, n2, lane);
  const float hi = numpy_pairwise_sum(a + n2, n - n2, lane);
  return __fadd_rn(lo, hi);
}

template <int K>
__global__ void __launch_bounds__(256)
gmm_cdf_kernel(const float* __restrict__ sigma, const float* __restrict__ mu, const float* __restrict__ wgt,
               int w_is_logits, int M, long n_pos, const int32_t* __restrict__ ch_list, int n_ch, int minmax,
               const int32_t* __restrict__ s_pair, const int32_t* __restrict__ s_minmax, long pair_stride,
               int row_pitch, int L_max, float scale_bound, const float* __restrict__ y_hat_nhwc,
               int32_t* __restrict__ rows, int32_t* __restrict__ intervals) {
  // element (pos, j) of stream j: channel ch_list[j] of pair s_pair[j] (0 without a table) under its own minmax
  extern __shared__ float cdf_smem[];             // [warps per block][L_max]: the clipped pmf of each warp's element
  const int warp_in_block = threadIdx.x >> 5;
  const long wid = (long)blockIdx.x * (blockDim.x >> 5) + warp_in_block;
  const int lane = threadIdx.x & 31;
  if (wid >= n_pos * n_ch) return;
  const long pos_w = wid / n_ch;
  const int j = (int)(wid - pos_w * n_ch);
  const int ch = ch_list[j];
  if (s_minmax) minmax = s_minmax[j];
  const long pos = (s_pair ? s_pair[j] * pair_stride : 0) + pos_w;
  const int L = 2 * minmax + 1;
  float* pmf = cdf_smem + (size_t)warp_in_block * L_max;
  float s_k[K], m_k[K], w_k[K];
  const long base = pos * (long)(M * K) + ch;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    s_k[k] = fmaxf(sigma[base + (long)k * M], scale_bound);             // lower_bound_scale (:1013)
    m_k[k] = __fadd_rn(mu[base + (long)k * M], (float)minmax);          // means + minmax (:1001)
    w_k[k] = wgt[base + (long)k * M];
  }
  if (w_is_logits) {                              // torch.softmax over K (MASIC.py:393): exp(x - max) / sum, fp32
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < K; ++k) mx = fmaxf(mx, w_k[k]);
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) { w_k[k] = expf(__fsub_rn(w_k[k], mx)); sum = __fadd_rn(sum, w_k[k]); }
#pragma unroll
    for (int k = 0; k < K; ++k) w_k[k] = __fdiv_rn(w_k[k], sum);
  }
  // pass 1: the clipped pmf (np.clip(pmf, 1/65536, 1)), one sample per lane and step
  for (int s = lane; s < L; s += 32) {
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float v = fabsf(__fsub_rn((float)s, m_k[k]));
      const float up = __fmul_rn(0.5f, erfcf(__fmul_rn(kInvSqrt2Neg, __fdiv_rn(__fsub_rn(0.5f, v), s_k[k]))));
      const float lo = __fmul_rn(0.5f, erfcf(__fmul_rn(kInvSqrt2Neg, __fdiv_rn(__fsub_rn(-0.5f, v), s_k[k]))));
      const float t = __fmul_rn(__fsub_rn(up, lo), w_k[k]);
      acc = (k == 0) ? t : __fadd_rn(acc, t);
    }
    pmf[s] = fminf(fmaxf(acc, 1.0f / 65536.0f), 1.0f);
  }
  __syncwarp();
  const float total = numpy_pairwise_sum(pmf, L, lane);
  // pass 2: rounded counts and their running sum, 32 samples at a time
  const int sym = y_hat_nhwc ? (int)y_hat_nhwc[pos * (long)M + ch] + minmax : -1;
  int run = 0, lo = 0, fr = 0;
  int32_t* row = rows ? rows + wid * (long)row_pitch : nullptr;
  if (row && lane == 0) row[0] = 0;
  for (int s0 = 0; s0 < L; s0 += 32) {
    const int s = s0 + lane;
    int c = 0;
    if (s < L) c = (int)rintf(__fmul_rn(__fdiv_rn(pmf[s], total), 65536.0f));
    int inc = c;                                  // inclusive scan inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (s < L) {
      if (row) row[s + 1] = run + inc;
      if (s == sym) { lo = run + inc - c; fr = c; }
    }
    run += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (intervals) {
    // the lane that saw the symbol holds (lo, fr); everyone else holds zeros
    lo = __reduce_add_sync(0xffffffffu, lo);
    fr = __reduce_add_sync(0xffffffffu, fr);
    if (lane == 0) {
      intervals[wid * 3 + 0] = lo;
      intervals[wid * 3 + 1] = fr;
      intervals[wid * 3 + 2] = run;
    }
  }
}

inline View mkview(int layout_nhwc, int C, int P) {
  View v;
  if (layout_nhwc) { v.sn = (long)C * P; v.sc = 1; v.sp = C; }
  else { v.sn = (long)C * P; v.sc = P; v.sp = 1; }
  return v;
}

}  // namespace

extern "C" int masic_gmm_likelihood_fwd(const float* y, const float* sigma, const float* mu,
                                        const float* weights, int weights_are_logits, int in_nhwc,
                                        int n, int m, int k, int hw, float scale_bound,
                                        float* y_hat, float* lik, int32_t* symbols, int out_nhwc,
                                        void* yq_bf16, int bf_pitch, int bf_coff,
                                        const float* rowscale, int rs_stride, int rs_off, int f16, void* stream) {
  if (!y || !sigma || !mu || !weights || n <= 0 || m <= 0 || hw <= 0) return MASIC_EINVAL;
  if (k != 5) return MASIC_ENOSUP;    // HSIC hard-codes K = 5 (MASIC.py:653, test2_real.py:395)
  const View vy = mkview(in_nhwc, m, hw), vp = mkview(in_nhwc, m * k, hw), vo = mkview(out_nhwc, m, hw);
  dim3 grid((hw + 31) / 32, (m + 31) / 32, n), block(32, 8);
  if (in_nhwc && weights_are_logits && !out_nhwc && y_hat && lik && !symbols && !yq_bf16 && (m % 4) == 0 &&
      (reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(sigma) | reinterpret_cast<uintptr_t>(mu) |
       reinterpret_cast<uintptr_t>(weights)) % 16 == 0) {
    gmm_fwd_nhwc_v4_kernel<5><<<grid, dim3(8, 32), 0, static_cast<cudaStream_t>(stream)>>>(
        y, sigma, mu, weights, m, hw, scale_bound, y_hat, lik);
    return (int)cudaGetLastError();
  }
  gmm_fwd_kernel<5><<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      y, vy, sigma, mu, weights, vp, weights_are_logits, in_nhwc, m, hw, scale_bound, y_hat, lik, vo,
      symbols, static_cast<__nv_bfloat16*>(yq_bf16), bf_pitch, bf_coff, f16, rowscale, rs_stride, rs_off);
  return (int)cudaGetLastError();
}

extern "C" int masic_gc_likelihood_fwd(const float* y, const float* scales, const float* means,
                                       int64_t numel, float scale_bound, float* y_hat, float* lik,
                                       int32_t* symbols, void* stream) {
  if (!y || numel < 0 || (lik && !scales)) return MASIC_EINVAL;
  if (numel == 0) return MASIC_OK;
  gc_fwd_kernel<<<(unsigned)((numel + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      y, scales, means, numel, scale_bound, y_hat, lik, symbols);
  return (int)cudaGetLastError();
}

extern "C" int masic_gc_build_indexes(const float* scales, int64_t numel, const float* scale_table,
                                      int table_len, float scale_bound, int32_t* indexes, void* stream) {
  if (!scales || !scale_table || !indexes || table_len <= 0 || table_len > 4096 || numel < 0)
    return MASIC_EINVAL;
  if (numel == 0) return MASIC_OK;
  gc_indexes_kernel<<<(unsigned)((numel + 255) / 256), 256, table_len * sizeof(float),
                      static_cast<cudaStream_t>(stream)>>>(scales, numel, scale_table, table_len,
                                                           scale_bound, indexes);
  return (int)cudaGetLastError();
}

extern "C" int masic_eb_fwd(const float* z, int in_nhwc, int n, int c, int hw,
                            const float* const* matrices, const float* const* biases,
                            const float* const* factors, const float* quantiles, float* z_hat,
                            float* lik, int32_t* symbols, int out_nhwc, void* zq_bf16, int bf_pitch,
                            int f16, void* stream) {
  if (!z || !matrices || !biases || !factors || !quantiles || n <= 0 || c <= 0 || hw <= 0)
    return MASIC_EINVAL;
  const View vz = mkview(in_nhwc, c, hw), vo = mkview(out_nhwc, c, hw);
  dim3 grid((hw + 255) / 256, c, n);
  eb_fwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      z, vz, hw, matrices[0], matrices[1], matrices[2], matrices[3], matrices[4], biases[0], biases[1],
      biases[2], biases[3], biases[4], factors[0], factors[1], factors[2], factors[3], quantiles, z_hat,
      lik, vo, symbols, static_cast<__nv_bfloat16*>(zq_bf16), bf_pitch, f16);
  return (int)cudaGetLastError();
}

extern "C" int masic_quantize(const float* x, const float* means, int64_t numel, float* dequantized,
                              int32_t* symbols, void* stream) {
  if (!x || numel < 0) return MASIC_EINVAL;
  if (numel == 0) return MASIC_OK;
  quantize_kernel<<<(unsigned)((numel + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, means, numel, dequantized, symbols);
  return (int)cudaGetLastError();
}

extern "C" int masic_latent_prep(const float* y_nhwc, int64_t n_pixels, int c, void* y_abs_bf16,
                                 int abs_pitch, void* y_round_bf16, int rnd_pitch, int rnd_coff,
                                 const float* rowscale, int rs_stride, int rs_off, int f16, void* stream) {
  if (!y_nhwc || n_pixels <= 0 || c <= 0) return MASIC_EINVAL;
  const long total = n_pixels * c;
  const bool v4 = (c & 3) == 0 && (abs_pitch & 3) == 0 && (rnd_pitch & 3) == 0 && (rnd_coff & 3) == 0;   // as in the kernel
  const long threads = v4 ? total / 4 : total;
  latent_prep_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      y_nhwc, total, c, static_cast<__nv_bfloat16*>(y_abs_bf16), abs_pitch,
      static_cast<__nv_bfloat16*>(y_round_bf16), rnd_pitch, rnd_coff, rowscale, rs_stride, rs_off, f16);
  return (int)cudaGetLastError();
}

// one launch of gmm_cdf_kernel: pmf rows of up to L_max = 2 * max_minmax + 1 floats per warp in shared memory
static int launch_gmm_cdfs(const float* sigma, const float* mu, const float* wgt, int w_is_logits, int m, int64_t n_pos,
                           const int32_t* ch_list, int n_ch, int minmax, const int32_t* s_pair, const int32_t* s_minmax,
                           int64_t pair_stride, int row_pitch, int max_minmax, float scale_bound, const float* y_hat,
                           int32_t* rows, int32_t* intervals, cudaStream_t stream) {
  const long warps = n_pos * n_ch;
  if (warps == 0) return MASIC_OK;
  const int L = 2 * max_minmax + 1;
  int wpb = 8;                                      // warps per block, limited by L floats of shared memory per warp
  while (wpb > 1 && (size_t)wpb * L * sizeof(float) > 96 * 1024) wpb >>= 1;
  const size_t smem = (size_t)wpb * L * sizeof(float);
  if (smem > 200 * 1024) return MASIC_ENOSUP;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(gmm_cdf_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  const long blocks = (warps + wpb - 1) / wpb;
  gmm_cdf_kernel<5><<<(unsigned)blocks, wpb * 32, smem, stream>>>(
      sigma, mu, wgt, w_is_logits, m, n_pos, ch_list, n_ch, minmax, s_pair, s_minmax, pair_stride, row_pitch, L,
      scale_bound, y_hat, rows, intervals);
  return (int)cudaGetLastError();
}

extern "C" int masic_gmm_symbol_cdfs(const float* sigma_nhwc, const float* mu_nhwc, const float* weights_nhwc,
                                     int weights_are_logits, int m, int k, int64_t n_pos,
                                     const int32_t* ch_list, int n_ch, int minmax, float scale_bound,
                                     const float* y_hat_nhwc, int32_t* rows, int32_t* intervals, void* stream) {
  if (!sigma_nhwc || !mu_nhwc || !weights_nhwc || !ch_list || m <= 0 || n_pos < 0 || n_ch < 0 || minmax < 1 ||
      minmax > 32767 || (!rows && !intervals) || (intervals && !y_hat_nhwc))
    return MASIC_EINVAL;
  if (k != 5) return MASIC_ENOSUP;
  return launch_gmm_cdfs(sigma_nhwc, mu_nhwc, weights_nhwc, weights_are_logits, m, n_pos, ch_list, n_ch, minmax, nullptr,
                         nullptr, 0, 2 * minmax + 2, minmax, scale_bound, y_hat_nhwc, rows, intervals,
                         static_cast<cudaStream_t>(stream));
}

extern "C" int masic_gmm_symbol_cdfs_pairs(const float* sigma_nhwc, const float* mu_nhwc, const float* weights_nhwc,
                                           int weights_are_logits, int m, int k, int64_t n_pos, int64_t pair_stride,
                                           const int32_t* stream_pair, const int32_t* stream_ch,
                                           const int32_t* stream_minmax, int n_streams, int max_minmax,
                                           float scale_bound, const float* y_hat_nhwc, int32_t* rows, int row_pitch,
                                           int32_t* intervals, void* stream) {
  if (!sigma_nhwc || !mu_nhwc || !weights_nhwc || !stream_pair || !stream_ch || !stream_minmax || m <= 0 ||
      n_pos < 0 || pair_stride < 0 || n_streams < 0 || max_minmax < 1 || max_minmax > 32767 || (!rows && !intervals) ||
      (intervals && !y_hat_nhwc) || (rows && row_pitch < 2 * max_minmax + 2))
    return MASIC_EINVAL;
  if (k != 5) return MASIC_ENOSUP;
  return launch_gmm_cdfs(sigma_nhwc, mu_nhwc, weights_nhwc, weights_are_logits, m, n_pos, stream_ch, n_streams, 0,
                         stream_pair, stream_minmax, pair_stride, row_pitch, max_minmax, scale_bound, y_hat_nhwc, rows,
                         intervals, static_cast<cudaStream_t>(stream));
}
