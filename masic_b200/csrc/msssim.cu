// msssim.cu — SSIM / MS-SSIM of two NCHW fp32 image batches, per (n, c) plane, on the device (sm_100a).
//
// Replaces (reference, file:line):
//   pytorch_msssim.ms_ssim(x_hat, x, data_range=1.0)   coremasic/mywork/test2_real.py:88-114 (the eval loop's
//   MS-SSIM column; test3_real.py reports the same after the enhancement net).  pytorch_msssim 1.0 runs 5 levels x
//   5 Gaussian-filtered maps x 2 separable grouped conv2d passes plus ~12 elementwise ops per level, each a full fp32
//   pass over HBM; here: one pooling launch per pyramid level, one statistics launch over every level, one final launch.
//
// Algorithm (pytorch_msssim 1.0, restated in float64 in oracle/msssim.py):
//   window: 11-tap Gaussian, sigma 1.5, float32 taps normalised to sum 1, separable valid correlation per channel;
//   mu_x = G(x), sigma_x^2 = G(x^2) - mu_x^2, sigma_xy = G(xy) - mu_x mu_y;
//   cs = (2 sigma_xy + C2) / (sigma_x^2 + sigma_y^2 + C2),  ssim = (2 mu_x mu_y + C1) / (mu_x^2 + mu_y^2 + C1) * cs;
//   levels 0..L-2 contribute relu(mean cs)^w_l, level L-1 contributes (relu of) mean ssim ^ w_{L-1};
//   between levels avg_pool2d(kernel 2, stride 2, padding (h % 2, w % 2), count_include_pad=True).
//
// Accuracy: x and y are shifted by data_range/2 before the products.  Variances and the covariance do not change and
// the luminance term adds the shift back, but G(x^2) - mu^2 no longer cancels the (large) square of the mean in fp32.
//
// Deterministic and batch invariant: every (level, plane, tile) block writes fp64 partial sums of its cs and ssim
// maps; the final launch adds each plane's partials in a fixed order that does not depend on the batch size.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/masic_b200.h"

namespace {

constexpr int WIN = 11;
constexpr int MAX_LEVELS = 5;
constexpr int TW = 32, TH = 48;                 // output tile of one statistics block
constexpr int PR = TH + WIN - 1;                // patch rows (58)
constexpr int PC = 44;                          // patch columns: TW + 10 = 42 used, padded for float4 reads
constexpr int HSEG = 4;                         // horizontal-pass outputs per thread (reads 16 patch columns)
constexpr int VSEG = 6;                         // vertical-pass outputs per thread
constexpr int ST_THREADS = 256;                 // = TW * TH / VSEG
constexpr int POOL_THREADS = 256;
constexpr size_t ST_SMEM = sizeof(float) * (2 * PR * PC + 5 * PR * TW);

static_assert(TW * (TH / VSEG) == ST_THREADS, "one vertical segment per thread");
static_assert(TW + WIN - 1 <= PC && (TW - HSEG) + 16 <= PC, "float4 patch reads stay inside a row");

struct Level {
  const float* x;
  const float* y;
  int h, w;               // level size; the maps are (h - 10) x (w - 10)
  int tiles_x, tiles;     // statistics tiles per plane
  int block0;             // first statistics block of this level
};

struct Args {
  Level lv[MAX_LEVELS];
  int levels, planes;
  float taps[WIN];
  float shift, c1, c2;
  double weights[MAX_LEVELS];
  int nonneg_last;
};

int level_size(int s, int l) {
  for (int i = 0; i < l; ++i) s = (s + (s & 1)) / 2;   // avg_pool2d(2, padding = s % 2): floor((s + 2 (s % 2)) / 2)
  return s;
}

size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

// avg_pool2d(kernel 2, stride 2, padding (h % 2, w % 2), count_include_pad=True) of x and y (blockIdx.y selects)
__global__ void __launch_bounds__(POOL_THREADS) msssim_pool_kernel(const float* __restrict__ x,
                                                                    const float* __restrict__ y, float* __restrict__ ox,
                                                                    float* __restrict__ oy, int planes, int h, int w,
                                                                    int ho, int wo) {
  const float* in = blockIdx.y ? y : x;
  float* out = blockIdx.y ? oy : ox;
  const int ph = h & 1, pw = w & 1;
  const long total = (long)planes * ho * wo;
  for (long i = (long)blockIdx.x * POOL_THREADS + threadIdx.x; i < total; i += (long)gridDim.x * POOL_THREADS) {
    const int j = (int)(i % wo);
    const long r = i / wo;
    const int k = (int)(r % ho);
    const float* src = in + (r / ho) * (long)h * w;
    float s = 0.f;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int iy = 2 * k - ph + a;
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const int ix = 2 * j - pw + b;
        if (iy >= 0 && iy < h && ix >= 0 && ix < w) s += __ldg(src + (long)iy * w + ix);
      }
    }
    out[i] = s / 4.f;
  }
}

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int wp = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[wp] = v;
  __syncthreads();
  double t = 0.0;
  if (wp == 0) {
    t = l < ST_THREADS / 32 ? sh[l] : 0.0;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;   // valid in thread 0
}

// One block = one TW x TH tile of one plane at one level.  partial[2 b + {0, 1}] = sums of the tile's {cs, ssim} maps.
__global__ void __launch_bounds__(ST_THREADS, 3) msssim_stats_kernel(const Args a, double* __restrict__ partial) {
  extern __shared__ float4 smem4[];
  float* px = reinterpret_cast<float*>(smem4);   // [PR][PC]  x - shift
  float* py = px + PR * PC;                      // [PR][PC]  y - shift
  float* hq = py + PR * PC;                      // [5][PR][TW]  horizontal pass of x, y, x^2, y^2, xy
  __shared__ double red[ST_THREADS / 32];

  const int b = blockIdx.x;
  int l = 0;
#pragma unroll
  for (int i = 1; i < MAX_LEVELS; ++i)
    if (i < a.levels && b >= a.lv[i].block0) l = i;
  const Level& L = a.lv[l];
  const int rel = b - L.block0;
  const int plane = rel / L.tiles, tile = rel - plane * L.tiles;
  const int oy = (tile / L.tiles_x) * TH, ox = (tile % L.tiles_x) * TW;
  const long poff = (long)plane * L.h * L.w;
  const float* __restrict__ xs = L.x + poff;
  const float* __restrict__ ys = L.y + poff;

  // all of a thread's loads are issued before the first store: one memory latency per block, not one per element
  constexpr int LOADS = (PR * PC + ST_THREADS - 1) / ST_THREADS;
  float lx[LOADS], ly[LOADS];
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    const int r = i / PC, c = i - r * PC;
    const int gy = oy + r, gx = ox + c;
    lx[k] = ly[k] = a.shift;
    if (i < PR * PC && gy < L.h && gx < L.w) {
      lx[k] = __ldg(xs + (long)gy * L.w + gx);
      ly[k] = __ldg(ys + (long)gy * L.w + gx);
    }
  }
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    if (i < PR * PC) {
      px[i] = lx[k] - a.shift;
      py[i] = ly[k] - a.shift;
    }
  }
  __syncthreads();

  // horizontal pass: HSEG consecutive outputs of one patch row per item
  for (int it = threadIdx.x; it < PR * (TW / HSEG); it += ST_THREADS) {
    const int r = it / (TW / HSEG), c0 = (it % (TW / HSEG)) * HSEG;
    const float4* rx = reinterpret_cast<const float4*>(px + r * PC + c0);
    const float4* ry = reinterpret_cast<const float4*>(py + r * PC + c0);
    float vx[16], vy[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 u = rx[q], v = ry[q];
      vx[4 * q] = u.x; vx[4 * q + 1] = u.y; vx[4 * q + 2] = u.z; vx[4 * q + 3] = u.w;
      vy[4 * q] = v.x; vy[4 * q + 1] = v.y; vy[4 * q + 2] = v.z; vy[4 * q + 3] = v.w;
    }
    float s[5][HSEG];
#pragma unroll
    for (int j = 0; j < HSEG; ++j) s[0][j] = s[1][j] = s[2][j] = s[3][j] = s[4][j] = 0.f;
#pragma unroll
    for (int k = 0; k < HSEG + WIN - 1; ++k) {
      const float xx = vx[k] * vx[k], yy = vy[k] * vy[k], xy = vx[k] * vy[k];
#pragma unroll
      for (int j = 0; j < HSEG; ++j) {
        const int t = k - j;
        if (t >= 0 && t < WIN) {
          const float g = a.taps[t];
          s[0][j] = fmaf(g, vx[k], s[0][j]);
          s[1][j] = fmaf(g, vy[k], s[1][j]);
          s[2][j] = fmaf(g, xx, s[2][j]);
          s[3][j] = fmaf(g, yy, s[3][j]);
          s[4][j] = fmaf(g, xy, s[4][j]);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q)
      *reinterpret_cast<float4*>(hq + (q * PR + r) * TW + c0) = make_float4(s[q][0], s[q][1], s[q][2], s[q][3]);
  }
  __syncthreads();

  // vertical pass: VSEG outputs of one column per thread, then cs / ssim per pixel
  const int col = threadIdx.x % TW, r0 = (threadIdx.x / TW) * VSEG;
  float m[5][VSEG];
#pragma unroll
  for (int j = 0; j < VSEG; ++j) m[0][j] = m[1][j] = m[2][j] = m[3][j] = m[4][j] = 0.f;
#pragma unroll
  for (int k = 0; k < VSEG + WIN - 1; ++k) {
    float v[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) v[q] = hq[(q * PR + r0 + k) * TW + col];
#pragma unroll
    for (int j = 0; j < VSEG; ++j) {
      const int t = k - j;
      if (t >= 0 && t < WIN) {
        const float g = a.taps[t];
#pragma unroll
        for (int q = 0; q < 5; ++q) m[q][j] = fmaf(g, v[q], m[q][j]);
      }
    }
  }
  const int ho = L.h - (WIN - 1), wo = L.w - (WIN - 1);
  float scs = 0.f, sss = 0.f;
  if (ox + col < wo) {
#pragma unroll
    for (int j = 0; j < VSEG; ++j) {
      if (oy + r0 + j < ho) {
        const float mx = m[0][j], my = m[1][j];                 // means of the shifted images
        const float vxx = m[2][j] - mx * mx, vyy = m[3][j] - my * my, vxy = m[4][j] - mx * my;
        const float ux = mx + a.shift, uy = my + a.shift;       // means of the images
        const float csn = 2.f * vxy + a.c2, csd = vxx + vyy + a.c2;
        const float ln = 2.f * ux * uy + a.c1, ld = ux * ux + uy * uy + a.c1;
        const float cs = csn / csd;
        scs += cs;
        sss += ln / ld * cs;
      }
    }
  }
  const double tcs = block_sum((double)scs, red);
  const double tss = block_sum((double)sss, red);
  if (threadIdx.x == 0) {
    partial[2 * (long)b] = tcs;
    partial[2 * (long)b + 1] = tss;
  }
}

// One block per plane, one warp per (level, map): lane-strided fixed-order sums of the tile partials, a fixed shuffle
// tree, then the weighted product in fp64.
__global__ void msssim_final_kernel(const Args a, const double* __restrict__ partial, float* __restrict__ out) {
  __shared__ double tot[MAX_LEVELS * 2];
  const int p = blockIdx.x, wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (wp < 2 * a.levels) {
    const Level& L = a.lv[wp >> 1];
    const double* src = partial + 2 * ((long)L.block0 + (long)p * L.tiles) + (wp & 1);
    double s = 0.0;
    for (int t = lane; t < L.tiles; t += 32) s += src[2 * t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) tot[wp] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 1.0;
    for (int l = 0; l < a.levels; ++l) {
      const double cnt = (double)(a.lv[l].h - (WIN - 1)) * (double)(a.lv[l].w - (WIN - 1));
      if (l < a.levels - 1) {
        v *= pow(fmax(tot[2 * l] / cnt, 0.0), a.weights[l]);
      } else {
        const double s = tot[2 * l + 1] / cnt;
        v *= pow(a.nonneg_last ? fmax(s, 0.0) : s, a.weights[l]);
      }
    }
    out[p] = (float)v;
  }
}

// scratch layout: pyramid levels 1..L-1 (x then y, each 256-byte aligned), then 2 doubles per statistics block
bool plan(int n, int c, int h, int w, int levels, Args* a, size_t* bytes) {
  if (n <= 0 || c <= 0 || h <= 0 || w <= 0 || levels < 1 || levels > MAX_LEVELS) return false;
  const long planes = (long)n * c;
  if (planes > (1L << 30)) return false;
  size_t off = 0;
  long blocks = 0;
  for (int l = 0; l < levels; ++l) {
    const int hl = level_size(h, l), wl = level_size(w, l);
    if (hl < WIN || wl < WIN) return false;
    Level& L = a->lv[l];
    L.h = hl;
    L.w = wl;
    L.tiles_x = (wl - (WIN - 1) + TW - 1) / TW;
    L.tiles = L.tiles_x * ((hl - (WIN - 1) + TH - 1) / TH);
    L.block0 = (int)blocks;
    blocks += planes * L.tiles;
    if (blocks > 0x7fffffffL) return false;
    if (l > 0) off += 2 * align256(sizeof(float) * planes * hl * wl);
  }
  a->levels = levels;
  a->planes = (int)planes;
  *bytes = off + sizeof(double) * 2 * blocks;
  return true;
}

// Window, constants and level weights of a call (the pyramid pointers are set by the caller).
void set_constants(Args* a, int levels, float data_range, float k1, float k2, const float* weights_host,
                   int nonneg_last) {
  // the window of pytorch_msssim's _fspecial_gauss_1d(11, 1.5), in float32 as the package computes it
  float g[WIN], gs = 0.f;
  for (int i = 0; i < WIN; ++i) {
    const float d = (float)(i - WIN / 2);
    g[i] = expf(-(d * d) / (2.f * 1.5f * 1.5f));
    gs += g[i];
  }
  for (int i = 0; i < WIN; ++i) a->taps[i] = g[i] / gs;
  a->shift = 0.5f * data_range;
  a->c1 = (k1 * data_range) * (k1 * data_range);
  a->c2 = (k2 * data_range) * (k2 * data_range);
  for (int l = 0; l < MAX_LEVELS; ++l) a->weights[l] = l < levels ? (double)weights_host[l] : 0.0;
  a->nonneg_last = nonneg_last ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------- backward
// d(sum over planes of MS-SSIM)/dx.  With m_l the mean of level l's map (cs, the last level's ssim) and
// V = prod_l relu(m_l)^w_l, dV/dm_l = w_l m_l^(w_l - 1) prod_{k != l} relu(m_k)^w_k, and 0 where relu clamps m_l (as
// torch's relu / prod backward give: a zero factor zeroes every level).  Per level, the map at p depends on x through
// mu_x = G(x), E[x^2] = G(x^2) and E[xy] = G(xy) at p, so
//   dm_l/dx(q) = (1 / cnt) (G^T a + 2 x G^T b + y G^T c)(q),   a, b, c = d map / d(mu_x, E[x^2], E[xy]) per pixel,
// with x, y shifted by data_range/2 like the forward (the shift is a constant: the gradient is the same).  Levels are
// joined through the transpose of the pooling: each fine pixel takes 1/4 of the one coarse cell whose window holds it.
//
// Launches: one coefficient launch (per plane and level: grad_scale dV/dm_l / cnt_l, from the forward's tile partials),
// one map launch over every level (the statistics grid, writing a, b, c), then one gather launch per level, coarsest
// first.  Every output element is a fixed-order gather of its plane's data: deterministic and batch invariant.

struct Bwd {
  float* map[MAX_LEVELS];     // level l: a, b, c, each planes x (h - 10) x (w - 10), mstride floats apart
  long mstride[MAX_LEVELS];
  float* grad[MAX_LEVELS];    // level l's gradient, planes x h x w (level 0: dx)
  const float* coef;          // [plane][MAX_LEVELS]: grad_scale * dV/dm_l / cnt_l
};

constexpr size_t GA_SMEM = sizeof(float) * (3 * PR * PC + 3 * PR * TW);

// One block per plane: the level sums in msssim_final_kernel's order, then the per-level coefficients in fp64.
__global__ void msssim_bwd_coef_kernel(const Args a, const double* __restrict__ partial, float grad_scale,
                                       float* __restrict__ coef) {
  __shared__ double tot[MAX_LEVELS * 2];
  const int p = blockIdx.x, wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (wp < 2 * a.levels) {
    const Level& L = a.lv[wp >> 1];
    const double* src = partial + 2 * ((long)L.block0 + (long)p * L.tiles) + (wp & 1);
    double s = 0.0;
    for (int t = lane; t < L.tiles; t += 32) s += src[2 * t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) tot[wp] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double m[MAX_LEVELS], f[MAX_LEVELS], cnt[MAX_LEVELS];
    bool clamps[MAX_LEVELS];
    for (int l = 0; l < a.levels; ++l) {
      cnt[l] = (double)(a.lv[l].h - (WIN - 1)) * (double)(a.lv[l].w - (WIN - 1));
      const bool last = l == a.levels - 1;
      m[l] = tot[2 * l + (last ? 1 : 0)] / cnt[l];
      clamps[l] = (!last || a.nonneg_last) && !(m[l] > 0.0);
      f[l] = pow(clamps[l] ? 0.0 : m[l], a.weights[l]);
    }
    for (int l = 0; l < MAX_LEVELS; ++l) {
      double d = 0.0;
      if (l < a.levels && !clamps[l]) {
        d = a.weights[l] * pow(m[l], a.weights[l] - 1.0);
        for (int k = 0; k < a.levels; ++k)
          if (k != l) d *= f[k];
        d = (double)grad_scale * d / cnt[l];
      }
      coef[p * MAX_LEVELS + l] = (float)d;
    }
  }
}

// The statistics grid again (the same loads and filter passes as msssim_stats_kernel, so the same filtered values);
// per output pixel it writes d map / d(mu_x, E[x^2], E[xy]) instead of summing the map.
__global__ void __launch_bounds__(ST_THREADS, 3) msssim_bwd_maps_kernel(const Args a, const Bwd bw) {
  extern __shared__ float4 smem4[];
  float* px = reinterpret_cast<float*>(smem4);   // [PR][PC]  x - shift
  float* py = px + PR * PC;                      // [PR][PC]  y - shift
  float* hq = py + PR * PC;                      // [5][PR][TW]  horizontal pass of x, y, x^2, y^2, xy

  const int b = blockIdx.x;
  int l = 0;
#pragma unroll
  for (int i = 1; i < MAX_LEVELS; ++i)
    if (i < a.levels && b >= a.lv[i].block0) l = i;
  const Level& L = a.lv[l];
  const int rel = b - L.block0;
  const int plane = rel / L.tiles, tile = rel - plane * L.tiles;
  const int oy = (tile / L.tiles_x) * TH, ox = (tile % L.tiles_x) * TW;
  const long poff = (long)plane * L.h * L.w;
  const float* __restrict__ xs = L.x + poff;
  const float* __restrict__ ys = L.y + poff;

  constexpr int LOADS = (PR * PC + ST_THREADS - 1) / ST_THREADS;
  float lx[LOADS], ly[LOADS];
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    const int r = i / PC, c = i - r * PC;
    const int gy = oy + r, gx = ox + c;
    lx[k] = ly[k] = a.shift;
    if (i < PR * PC && gy < L.h && gx < L.w) {
      lx[k] = __ldg(xs + (long)gy * L.w + gx);
      ly[k] = __ldg(ys + (long)gy * L.w + gx);
    }
  }
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    if (i < PR * PC) {
      px[i] = lx[k] - a.shift;
      py[i] = ly[k] - a.shift;
    }
  }
  __syncthreads();

  for (int it = threadIdx.x; it < PR * (TW / HSEG); it += ST_THREADS) {
    const int r = it / (TW / HSEG), c0 = (it % (TW / HSEG)) * HSEG;
    const float4* rx = reinterpret_cast<const float4*>(px + r * PC + c0);
    const float4* ry = reinterpret_cast<const float4*>(py + r * PC + c0);
    float vx[16], vy[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 u = rx[q], v = ry[q];
      vx[4 * q] = u.x; vx[4 * q + 1] = u.y; vx[4 * q + 2] = u.z; vx[4 * q + 3] = u.w;
      vy[4 * q] = v.x; vy[4 * q + 1] = v.y; vy[4 * q + 2] = v.z; vy[4 * q + 3] = v.w;
    }
    float s[5][HSEG];
#pragma unroll
    for (int j = 0; j < HSEG; ++j) s[0][j] = s[1][j] = s[2][j] = s[3][j] = s[4][j] = 0.f;
#pragma unroll
    for (int k = 0; k < HSEG + WIN - 1; ++k) {
      const float xx = vx[k] * vx[k], yy = vy[k] * vy[k], xy = vx[k] * vy[k];
#pragma unroll
      for (int j = 0; j < HSEG; ++j) {
        const int t = k - j;
        if (t >= 0 && t < WIN) {
          const float g = a.taps[t];
          s[0][j] = fmaf(g, vx[k], s[0][j]);
          s[1][j] = fmaf(g, vy[k], s[1][j]);
          s[2][j] = fmaf(g, xx, s[2][j]);
          s[3][j] = fmaf(g, yy, s[3][j]);
          s[4][j] = fmaf(g, xy, s[4][j]);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q)
      *reinterpret_cast<float4*>(hq + (q * PR + r) * TW + c0) = make_float4(s[q][0], s[q][1], s[q][2], s[q][3]);
  }
  __syncthreads();

  const int col = threadIdx.x % TW, r0 = (threadIdx.x / TW) * VSEG;
  float m[5][VSEG];
#pragma unroll
  for (int j = 0; j < VSEG; ++j) m[0][j] = m[1][j] = m[2][j] = m[3][j] = m[4][j] = 0.f;
#pragma unroll
  for (int k = 0; k < VSEG + WIN - 1; ++k) {
    float v[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) v[q] = hq[(q * PR + r0 + k) * TW + col];
#pragma unroll
    for (int j = 0; j < VSEG; ++j) {
      const int t = k - j;
      if (t >= 0 && t < WIN) {
        const float g = a.taps[t];
#pragma unroll
        for (int q = 0; q < 5; ++q) m[q][j] = fmaf(g, v[q], m[q][j]);
      }
    }
  }
  const int ho = L.h - (WIN - 1), wo = L.w - (WIN - 1);
  if (ox + col >= wo) return;
  const bool last = l == a.levels - 1;
  float* __restrict__ ma = bw.map[l] + (long)plane * ho * wo + ox + col;
  const long ms = bw.mstride[l];
#pragma unroll
  for (int j = 0; j < VSEG; ++j) {
    const int row = oy + r0 + j;
    if (row < ho) {
      const float mx = m[0][j], my = m[1][j];
      const float vxx = m[2][j] - mx * mx, vyy = m[3][j] - my * my, vxy = m[4][j] - mx * my;
      const float csn = 2.f * vxy + a.c2, csd = 1.f / (vxx + vyy + a.c2);
      const float cs = csn * csd;
      float db = -cs * csd;                               // d cs / d var_x    (= d cs / d E[x^2])
      float dc = 2.f * csd;                               // d cs / d cov_xy   (= d cs / d E[xy])
      float da = -2.f * mx * db - my * dc;                // d cs / d mu_x through var_x and cov_xy
      if (last) {                                         // ssim = lum * cs
        const float ux = mx + a.shift, uy = my + a.shift;
        const float ln = 2.f * ux * uy + a.c1, ld = 1.f / (ux * ux + uy * uy + a.c1);
        const float lum = ln * ld;
        const float dlum = 2.f * (uy - lum * ux) * ld;    // d lum / d mu_x
        da = lum * da + cs * dlum;
        db *= lum;
        dc *= lum;
      }
      float* o = ma + (long)row * wo;
      o[0] = da;
      o[ms] = db;
      o[2 * ms] = dc;
    }
  }
}

// Level l's gradient over TW x TH output pixels of one plane: G^T of the three coefficient maps (zero outside the
// valid maps), combined with x and y, scaled by the level's coefficient, plus 1/4 of the coarser level's gradient at the
// pooling cell that holds the pixel; level 0 adds `addend` (which may be dx itself).
__global__ void __launch_bounds__(ST_THREADS, 3) msssim_bwd_gather_kernel(const Args a, const Bwd bw, int l,
                                                                          const float* addend) {
  extern __shared__ float4 smem4[];
  float* pm = reinterpret_cast<float*>(smem4);   // [3][PR][PC]  maps, rows oy - 10 .., columns ox - 10 ..
  float* hq = pm + 3 * PR * PC;                  // [3][PR][TW]  horizontal pass

  const Level& L = a.lv[l];
  const int tiles_x = (L.w + TW - 1) / TW, tiles = tiles_x * ((L.h + TH - 1) / TH);
  const int plane = blockIdx.x / tiles, tile = blockIdx.x - plane * tiles;
  const int oy = (tile / tiles_x) * TH, ox = (tile % tiles_x) * TW;
  const int ho = L.h - (WIN - 1), wo = L.w - (WIN - 1);
  const long ms = bw.mstride[l];
  const float* __restrict__ src = bw.map[l] + (long)plane * ho * wo;

  constexpr int LOADS = (PR * PC + ST_THREADS - 1) / ST_THREADS;
  float lv[3][LOADS];
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    const int r = i / PC, c = i - r * PC;
    const int gy = oy - (WIN - 1) + r, gx = ox - (WIN - 1) + c;
    lv[0][k] = lv[1][k] = lv[2][k] = 0.f;
    if (i < PR * PC && gy >= 0 && gy < ho && gx >= 0 && gx < wo) {
      const float* p = src + (long)gy * wo + gx;
      lv[0][k] = __ldg(p);
      lv[1][k] = __ldg(p + ms);
      lv[2][k] = __ldg(p + 2 * ms);
    }
  }
#pragma unroll
  for (int k = 0; k < LOADS; ++k) {
    const int i = threadIdx.x + k * ST_THREADS;
    if (i < PR * PC) {
#pragma unroll
      for (int q = 0; q < 3; ++q) pm[q * PR * PC + i] = lv[q][k];
    }
  }
  __syncthreads();

  // horizontal pass of G^T: out(j) = sum_t g[10 - t] map(j - 10 + t), i.e. patch columns j .. j + 10
  for (int it = threadIdx.x; it < 3 * PR * (TW / HSEG); it += ST_THREADS) {
    const int q = it / (PR * (TW / HSEG)), rem = it - q * (PR * (TW / HSEG));
    const int r = rem / (TW / HSEG), c0 = (rem % (TW / HSEG)) * HSEG;
    const float4* rv = reinterpret_cast<const float4*>(pm + (q * PR + r) * PC + c0);
    float v[16];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4 t4 = rv[u];
      v[4 * u] = t4.x; v[4 * u + 1] = t4.y; v[4 * u + 2] = t4.z; v[4 * u + 3] = t4.w;
    }
    float s[HSEG];
#pragma unroll
    for (int j = 0; j < HSEG; ++j) s[j] = 0.f;
#pragma unroll
    for (int k = 0; k < HSEG + WIN - 1; ++k) {
#pragma unroll
      for (int j = 0; j < HSEG; ++j) {
        const int t = k - j;
        if (t >= 0 && t < WIN) s[j] = fmaf(a.taps[WIN - 1 - t], v[k], s[j]);
      }
    }
    *reinterpret_cast<float4*>(hq + (q * PR + r) * TW + c0) = make_float4(s[0], s[1], s[2], s[3]);
  }
  __syncthreads();

  const int col = threadIdx.x % TW, r0 = (threadIdx.x / TW) * VSEG;
  float m[3][VSEG];
#pragma unroll
  for (int j = 0; j < VSEG; ++j) m[0][j] = m[1][j] = m[2][j] = 0.f;
#pragma unroll
  for (int k = 0; k < VSEG + WIN - 1; ++k) {
    float v[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) v[q] = hq[(q * PR + r0 + k) * TW + col];
#pragma unroll
    for (int j = 0; j < VSEG; ++j) {
      const int t = k - j;
      if (t >= 0 && t < WIN) {
        const float g = a.taps[WIN - 1 - t];
#pragma unroll
        for (int q = 0; q < 3; ++q) m[q][j] = fmaf(g, v[q], m[q][j]);
      }
    }
  }
  const int ix = ox + col;
  if (ix >= L.w) return;
  const float kl = bw.coef[plane * MAX_LEVELS + l];
  const bool coarse = l + 1 < a.levels;
  const int hc = coarse ? a.lv[l + 1].h : 0, wc = coarse ? a.lv[l + 1].w : 0;
  const float* gc = coarse ? bw.grad[l + 1] + (long)plane * hc * wc + (ix + (L.w & 1)) / 2 : nullptr;
  const long poff = (long)plane * L.h * L.w;
#pragma unroll
  for (int j = 0; j < VSEG; ++j) {
    const int iy = oy + r0 + j;
    if (iy < L.h) {
      const long e = poff + (long)iy * L.w + ix;
      const float xv = __ldg(L.x + e) - a.shift, yv = __ldg(L.y + e) - a.shift;
      float g = kl * (m[0][j] + 2.f * xv * m[1][j] + yv * m[2][j]);
      if (coarse) g += 0.25f * gc[(long)((iy + (L.h & 1)) / 2) * wc];
      if (l == 0 && addend) g += addend[e];
      bw.grad[l][e] = g;
    }
  }
}

// work layout: coefficients, then per level the three coefficient maps, then the gradients of levels 1..L-1
bool plan_bwd(const Args& a, size_t* coef_bytes, size_t map_bytes[MAX_LEVELS], size_t grad_bytes[MAX_LEVELS],
              size_t* total) {
  *coef_bytes = align256(sizeof(float) * (size_t)a.planes * MAX_LEVELS);
  size_t t = *coef_bytes;
  for (int l = 0; l < a.levels; ++l) {
    map_bytes[l] = align256(sizeof(float) * (size_t)a.planes * (a.lv[l].h - (WIN - 1)) * (a.lv[l].w - (WIN - 1)));
    grad_bytes[l] = l ? align256(sizeof(float) * (size_t)a.planes * a.lv[l].h * a.lv[l].w) : 0;
    t += 3 * map_bytes[l] + grad_bytes[l];
  }
  // the gather grid of level 0 must fit one launch dimension
  const long tiles0 = (long)((a.lv[0].w + TW - 1) / TW) * ((a.lv[0].h + TH - 1) / TH);
  if (tiles0 * a.planes > 0x7fffffffL) return false;
  *total = t;
  return true;
}

}  // namespace

extern "C" int64_t masic_ms_ssim_scratch_bytes(int n, int c, int h, int w, int levels) {
  Args a;
  size_t bytes;
  if (!plan(n, c, h, w, levels, &a, &bytes)) return MASIC_EINVAL;
  return (int64_t)bytes;
}

extern "C" int masic_ms_ssim(const float* x, const float* y, int n, int c, int h, int w, int levels, float data_range,
                             float k1, float k2, const float* weights_host, int nonneg_last, void* scratch,
                             float* out_nc, void* stream) {
  if (!x || !y || !weights_host || !scratch || !out_nc) return MASIC_EINVAL;
  if (!(data_range > 0.f) || !(k1 >= 0.f) || !(k2 >= 0.f)) return MASIC_EINVAL;
  Args a;
  size_t bytes;
  if (!plan(n, c, h, w, levels, &a, &bytes)) return MASIC_EINVAL;
  set_constants(&a, levels, data_range, k1, k2, weights_host, nonneg_last);

  cudaStream_t s = static_cast<cudaStream_t>(stream);
  char* base = static_cast<char*>(scratch);
  a.lv[0].x = x;
  a.lv[0].y = y;
  size_t off = 0;
  for (int l = 1; l < levels; ++l) {
    const size_t lb = align256(sizeof(float) * a.planes * a.lv[l].h * a.lv[l].w);
    float* lx = reinterpret_cast<float*>(base + off);
    float* ly = reinterpret_cast<float*>(base + off + lb);
    off += 2 * lb;
    const long total = (long)a.planes * a.lv[l].h * a.lv[l].w;
    const int grid = (int)((total + POOL_THREADS - 1) / POOL_THREADS < 1184 ? (total + POOL_THREADS - 1) / POOL_THREADS
                                                                           : 1184);
    msssim_pool_kernel<<<dim3(grid, 2), POOL_THREADS, 0, s>>>(a.lv[l - 1].x, a.lv[l - 1].y, lx, ly, a.planes,
                                                             a.lv[l - 1].h, a.lv[l - 1].w, a.lv[l].h, a.lv[l].w);
    a.lv[l].x = lx;
    a.lv[l].y = ly;
  }
  double* partial = reinterpret_cast<double*>(base + off);
  // set per call: the attribute is per device, and a caller may alternate devices
  const cudaError_t e = cudaFuncSetAttribute(msssim_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)ST_SMEM);
  if (e != cudaSuccess) return (int)e;
  const int blocks = a.lv[levels - 1].block0 + a.planes * a.lv[levels - 1].tiles;
  msssim_stats_kernel<<<blocks, ST_THREADS, ST_SMEM, s>>>(a, partial);
  msssim_final_kernel<<<a.planes, 32 * 2 * levels, 0, s>>>(a, partial, out_nc);
  return (int)cudaGetLastError();
}

extern "C" int64_t masic_ms_ssim_bwd_work_bytes(int n, int c, int h, int w, int levels) {
  Args a;
  size_t bytes, coef_bytes, total, map_bytes[MAX_LEVELS], grad_bytes[MAX_LEVELS];
  if (!plan(n, c, h, w, levels, &a, &bytes)) return MASIC_EINVAL;
  if (!plan_bwd(a, &coef_bytes, map_bytes, grad_bytes, &total)) return MASIC_EINVAL;
  return (int64_t)total;
}

extern "C" int masic_ms_ssim_bwd(const float* x, const float* y, int n, int c, int h, int w, int levels,
                                 float data_range, float k1, float k2, const float* weights_host, int nonneg_last,
                                 const void* fwd_scratch, float grad_scale, const float* addend, float* dx, void* work,
                                 void* stream) {
  if (!x || !y || !weights_host || !fwd_scratch || !dx || !work) return MASIC_EINVAL;
  if (!(data_range > 0.f) || !(k1 >= 0.f) || !(k2 >= 0.f)) return MASIC_EINVAL;
  Args a;
  size_t bytes, coef_bytes, total, map_bytes[MAX_LEVELS], grad_bytes[MAX_LEVELS];
  if (!plan(n, c, h, w, levels, &a, &bytes)) return MASIC_EINVAL;
  if (!plan_bwd(a, &coef_bytes, map_bytes, grad_bytes, &total)) return MASIC_EINVAL;
  set_constants(&a, levels, data_range, k1, k2, weights_host, nonneg_last);

  // the forward's pyramid and tile partials, at the offsets masic_ms_ssim wrote them
  const char* fs = static_cast<const char*>(fwd_scratch);
  a.lv[0].x = x;
  a.lv[0].y = y;
  size_t off = 0;
  for (int l = 1; l < levels; ++l) {
    const size_t lb = align256(sizeof(float) * a.planes * a.lv[l].h * a.lv[l].w);
    a.lv[l].x = reinterpret_cast<const float*>(fs + off);
    a.lv[l].y = reinterpret_cast<const float*>(fs + off + lb);
    off += 2 * lb;
  }
  const double* partial = reinterpret_cast<const double*>(fs + off);

  Bwd bw = {};
  char* wb = static_cast<char*>(work);
  float* coef = reinterpret_cast<float*>(wb);
  bw.coef = coef;
  size_t woff = coef_bytes;
  for (int l = 0; l < levels; ++l) {
    bw.map[l] = reinterpret_cast<float*>(wb + woff);
    bw.mstride[l] = (long)(map_bytes[l] / sizeof(float));
    woff += 3 * map_bytes[l];
  }
  bw.grad[0] = dx;
  for (int l = 1; l < levels; ++l) {
    bw.grad[l] = reinterpret_cast<float*>(wb + woff);
    woff += grad_bytes[l];
  }

  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaFuncSetAttribute(msssim_bwd_maps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)ST_SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(msssim_bwd_gather_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GA_SMEM);
  if (e != cudaSuccess) return (int)e;
  msssim_bwd_coef_kernel<<<a.planes, 32 * 2 * levels, 0, s>>>(a, partial, grad_scale, coef);
  const int blocks = a.lv[levels - 1].block0 + a.planes * a.lv[levels - 1].tiles;
  msssim_bwd_maps_kernel<<<blocks, ST_THREADS, ST_SMEM, s>>>(a, bw);
  for (int l = levels - 1; l >= 0; --l) {
    const int tiles = ((a.lv[l].w + TW - 1) / TW) * ((a.lv[l].h + TH - 1) / TH);
    msssim_bwd_gather_kernel<<<a.planes * tiles, ST_THREADS, GA_SMEM, s>>>(a, bw, l, l == 0 ? addend : nullptr);
  }
  return (int)cudaGetLastError();
}
