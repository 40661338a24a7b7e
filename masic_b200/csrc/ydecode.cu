// ydecode.cu — device side of the wavefront y decoder (SURVEY §8(f)#3; MASIC.py:1227-1301, :1321-1384).
//
// The reference decodes one latent position at a time in Python: crop the decoded latents, run the context conv and
// the parameter nets, build one integer CDF per non-zero channel, ask the range decoder for the symbol, write it back.
// Here a WAVE of positions (t = w + 3h: their mask-A 5x5 contexts only reach earlier waves) is decoded per step, and
// nothing leaves the device inside a wave:
//   wave_gather_kernel     5x5 crops of the decoded latents + the per-position inputs of the parameter nets
//   (conv_tc plans)        context conv on the crops, parameter nets on the wave's positions   [bitstream.py]
//   wave_center_kernel     centre pixel of every crop's context output -> parameter-net input
//   gmm_cdf_kernel         the integer CDF row of every (position, channel)                    [entropy.cu]
//   range_decode_wave      one warp per CHANNEL STREAM walks the wave's positions: interval search in the CDF row
//                          (ballot over 32 entries at a time), range-coder update, the symbol written straight into the
//                          fp32 latent tensor and the zero-padded 16-bit copy the next waves' crops read.
// For this the y payload is split into one range-coded stream per (view, non-zero channel) — "format 2" of bitstream.py;
// the arithmetic of a stream is exactly csrc/cdf.cu's host coder (32-bit range, carry-less byte renormalisation), so
// the host encoder writes what this decoder reads and the host decoder (masic_range_decode_rows) reads it too.
#include <cuda_runtime.h>
#include <stdint.h>

#include <thread>
#include <vector>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"

namespace {

// Pair b of n_pairs, wave position i < n -> row r = b * n_max + i of the wave's buffers (pair b's tensors follow pair
// b - 1's; h16 only sets those pair strides):
// crop[r][dy][dx][:] = ypad_b[(h_i + dy) * (w16 + 4) + w_i + dx][:]   (16-bit, m channels = m / 8 uint4)
// rs[r][dy][dx][0:3] = mw_b[h_i * w16 + w_i][0:3]                      (right view: the mask weights of the position)
// px[r][0 : c_lo] = gmm_in_b[pos][0 : c_lo];  px[r][c_hi0 : cin] = gmm_in_b[pos][c_hi0 : cin]   (c_hi0 == cin: nothing)
__global__ void __launch_bounds__(256)
wave_gather_kernel(const uint4* __restrict__ ypad, int h16, int w16, int m8, const uint4* __restrict__ gmm_in, int cin8,
                   int c_lo8, int c_hi8, const float* __restrict__ mw, const int2* __restrict__ pos, int n, int n_pairs,
                   int n_max, uint4* __restrict__ crop, float* __restrict__ rs, uint4* __restrict__ px) {
  const int per_pos = 25 * m8 + cin8;
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n_pairs * n * per_pos) return;
  const int b = (int)(i / ((long)n * per_pos));
  const long ib = i - (long)b * n * per_pos;
  const int pi = (int)(ib / per_pos), r = (int)(ib - (long)pi * per_pos);
  const long row = (long)b * n_max + pi;
  const long plane = (long)h16 * w16;
  const int2 hw = pos[pi];
  if (r < 25 * m8) {
    const int pix = r / m8, c = r - pix * m8, dy = pix / 5, dx = pix - dy * 5;
    const uint4* yp = ypad + (long)b * (h16 + 4) * (w16 + 4) * m8;
    crop[row * 25 * m8 + r] = yp[((long)(hw.x + dy) * (w16 + 4) + hw.y + dx) * m8 + c];
    if (rs && c == 0) {
      const float* s = mw + (b * plane + (long)hw.x * w16 + hw.y) * 3;
      float* d = rs + (row * 25 + pix) * 3;
      d[0] = s[0]; d[1] = s[1]; d[2] = s[2];
    }
  } else {
    const int c = r - 25 * m8;
    if (c < c_lo8 || c >= c_hi8) px[row * cin8 + c] = gmm_in[(b * plane + (long)hw.x * w16 + hw.y) * cin8 + c];
  }
}

// px[i][c0 : c0 + nc] = ctx_out[i][2][2][c0 : c0 + nc]
__global__ void __launch_bounds__(256)
wave_center_kernel(const uint4* __restrict__ ctx_out, int cin8, int c08, int nc8, int n, uint4* __restrict__ px) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= (long)n * nc8) return;
  const int pi = (int)(i / nc8), c = (int)(i - (long)pi * nc8) + c08;
  px[(long)pi * cin8 + c] = ctx_out[((long)pi * 25 + 12) * cin8 + c];
}

struct StreamState { uint32_t range, code; uint32_t pos, pad; };

__global__ void range_streams_init_kernel(const uint8_t* __restrict__ data, const int64_t* __restrict__ offs, int n_streams,
                                          StreamState* __restrict__ st) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  const uint8_t* d = data + offs[s];
  const int64_t len = offs[s + 1] - offs[s];
  uint32_t code = 0;
  for (int i = 1; i <= 4; ++i) code = (code << 8) | (i < len ? d[i] : 0u);     // byte 0 is the encoder's initial cache (0)
  st[s].range = 0xFFFFFFFFu;
  st[s].code = code;
  st[s].pos = 5;
}

// One warp per stream.  rows: (n, n_streams, row_pitch) int32 CDF rows of the wave; the row of stream s has
// L1 = 2 * minmax_s + 2 entries, row[0] = 0, row[L1-1] = total.  Stream s codes channel ch_list[s] of pair s_pair[s]
// under minmax s_minmax[s] (without the tables: pair 0, the one minmax).  h16 only sets the pair strides.
__global__ void __launch_bounds__(128)
range_decode_wave_kernel(const int32_t* __restrict__ rows, int n, int n_streams, int row_pitch,
                         StreamState* __restrict__ st, const uint8_t* __restrict__ data,
                         const int64_t* __restrict__ offs, const int32_t* __restrict__ ch_list, int minmax,
                         const int32_t* __restrict__ s_pair, const int32_t* __restrict__ s_minmax,
                         const int2* __restrict__ pos, int h16, int w16, int M, float* __restrict__ y_nhwc,
                         uint16_t* __restrict__ ypad, int f16, int* __restrict__ error) {
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (s >= n_streams) return;
  const int ch = ch_list[s];
  if (s_minmax) minmax = s_minmax[s];
  const int L1 = 2 * minmax + 2;
  const long b = s_pair ? s_pair[s] : 0;
  float* yb = y_nhwc + b * h16 * w16 * M;
  uint16_t* ypb = ypad + b * (h16 + 4) * (w16 + 4) * M;
  const uint8_t* d = data + offs[s];
  const uint32_t len = (uint32_t)(offs[s + 1] - offs[s]);
  uint32_t range = st[s].range, code = st[s].code, bp = st[s].pos;
  for (int i = 0; i < n; ++i) {
    const int32_t* row = rows + ((long)i * n_streams + s) * row_pitch;
    const uint32_t total = (uint32_t)row[L1 - 1];
    if (total == 0u || total > (1u << 22)) { if (lane == 0) atomicExch(error, 1); return; }
    const uint32_t r = range / total;
    uint32_t v = code / r;
    if (v >= total) v = total - 1;
    // largest sym with row[sym] <= v: scan 32 entries at a time for the first entry > v (row is non-decreasing)
    int sym = -1;
    uint32_t cum = 0, nxt = 0;
    for (int s0 = 0; s0 < L1; s0 += 32) {
      const int j = s0 + lane;
      const uint32_t val = j < L1 ? (uint32_t)row[j] : 0xFFFFFFFFu;
      const unsigned ball = __ballot_sync(0xffffffffu, val > v);
      if (ball) {
        const int first = __ffs(ball) - 1;                    // row[s0 + first] is the first entry > v
        nxt = __shfl_sync(0xffffffffu, val, first);
        sym = s0 + first - 1;
        cum = first > 0 ? __shfl_sync(0xffffffffu, val, first - 1) : (uint32_t)row[s0 - 1];   // s0 >= 32 when first == 0
        break;
      }
    }
    if (sym < 0) { if (lane == 0) atomicExch(error, 2); return; }
    const uint32_t freq = nxt - cum;
    code -= r * cum;
    range = r * freq;
    while (range < (1u << 24)) {
      code = (code << 8) | (bp < len ? (uint32_t)d[bp] : 0u);
      ++bp;
      range <<= 8;
    }
    if (lane == 0) {
      const int2 hw = pos[i];
      const float val = (float)(sym - minmax);
      yb[((long)hw.x * w16 + hw.y) * M + ch] = val;
      ypb[((long)(hw.x + 2) * (w16 + 4) + hw.y + 2) * M + ch] = masic::pack16(val, f16);
    }
  }
  if (lane == 0) { st[s].range = range; st[s].code = code; st[s].pos = bp; }
}

// host range coder (identical arithmetic to csrc/cdf.cu's RangeEnc)
struct Enc {
  uint64_t low = 0;
  uint32_t range = 0xFFFFFFFFu;
  uint8_t cache = 0;
  int64_t cache_size = 1;
  std::vector<uint8_t> out;
  void shift_low() {
    if (static_cast<uint32_t>(low) < 0xFF000000u || (low >> 32) != 0) {
      uint8_t c = cache;
      do { out.push_back(static_cast<uint8_t>(c + static_cast<uint8_t>(low >> 32))); c = 0xFF; } while (--cache_size != 0);
      cache = static_cast<uint8_t>(low >> 24);
    }
    ++cache_size;
    low = (low & 0x00FFFFFFu) << 8;
  }
  void encode(uint32_t cum, uint32_t freq, uint32_t total) {
    const uint32_t r = range / total;
    low += static_cast<uint64_t>(r) * cum;
    range = r * freq;
    while (range < (1u << 24)) { range <<= 8; shift_low(); }
  }
  void finish() { for (int i = 0; i < 5; ++i) shift_low(); }
};

// The same coder on the device, one thread per stream: stream s codes intervals[(base[s] + i * stride[s]) * 3 ...]
// for i < n_pos into its own slot of slot_cap bytes.  An interval the host coder rejects sets *error = 1, a slot that
// would overflow *error = 2; the stream stops there.
__global__ void __launch_bounds__(128)
range_encode_streams_kernel(const int32_t* __restrict__ intervals, const int64_t* __restrict__ base,
                            const int64_t* __restrict__ stride, int64_t n_pos, int n_streams, uint8_t* __restrict__ slots,
                            int64_t slot_cap, int64_t* __restrict__ lens, int* __restrict__ error) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  uint8_t* out = slots + (int64_t)s * slot_cap;
  int64_t n_out = 0;
  uint64_t low = 0;
  uint32_t range = 0xFFFFFFFFu;
  uint8_t cache = 0;
  int64_t cache_size = 1;
  bool ok = true;
  auto shift_low = [&]() {
    if (static_cast<uint32_t>(low) < 0xFF000000u || (low >> 32) != 0) {
      if (n_out + cache_size > slot_cap) { ok = false; atomicExch(error, 2); }
      uint8_t c = cache;
      do { if (ok) out[n_out++] = static_cast<uint8_t>(c + static_cast<uint8_t>(low >> 32)); c = 0xFF; } while (--cache_size != 0);
      cache = static_cast<uint8_t>(low >> 24);
    }
    ++cache_size;
    low = (low & 0x00FFFFFFu) << 8;
  };
  const int32_t* iv = intervals + base[s] * 3;
  const int64_t step = stride[s] * 3;
  for (int64_t i = 0; i < n_pos && ok; ++i, iv += step) {
    const int32_t cum = iv[0], freq = iv[1], total = iv[2];
    if (cum < 0 || freq <= 0 || total <= 0 || (int64_t)cum + freq > total || total > (1 << 22)) {
      atomicExch(error, 1);
      ok = false;
      break;
    }
    const uint32_t r = static_cast<uint32_t>(range) / static_cast<uint32_t>(total);
    low += static_cast<uint64_t>(r) * static_cast<uint32_t>(cum);
    range = r * static_cast<uint32_t>(freq);
    while (range < (1u << 24)) { range <<= 8; shift_low(); }
  }
  for (int i = 0; i < 5 && ok; ++i) shift_low();
  lens[s] = n_out;
}

// offsets[0] = 0, offsets[s + 1] = lens[0] + ... + lens[s]: one block, each thread a contiguous run of streams
__global__ void __launch_bounds__(1024)
stream_offsets_kernel(const int64_t* __restrict__ lens, int n_streams, int64_t* __restrict__ offsets) {
  __shared__ int64_t part[1024];
  const int t = threadIdx.x;
  const int per = (n_streams + 1023) / 1024;
  const int s0 = min(t * per, n_streams), s1 = min(s0 + per, n_streams);
  int64_t sum = 0;
  for (int s = s0; s < s1; ++s) sum += lens[s];
  part[t] = sum;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {            // inclusive scan of the per-thread sums
    const int64_t v = t >= o ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int64_t run = part[t] - sum;
  if (t == 0) offsets[0] = 0;
  for (int s = s0; s < s1; ++s) { run += lens[s]; offsets[s + 1] = run; }
}

// packed[offsets[s] ...] = slot s, one block per stream
__global__ void __launch_bounds__(256)
pack_streams_kernel(const uint8_t* __restrict__ slots, int64_t slot_cap, const int64_t* __restrict__ offsets,
                    uint8_t* __restrict__ packed) {
  const int s = blockIdx.x;
  const uint8_t* src = slots + (int64_t)s * slot_cap;
  uint8_t* dst = packed + offsets[s];
  const int64_t len = offsets[s + 1] - offsets[s];
  for (int64_t i = threadIdx.x; i < len; i += blockDim.x) dst[i] = src[i];
}

}  // namespace

static int launch_wave_gather(const void* ypad16, int h16, int w16, int m, const void* gmm_in16, int cin, int c_lo,
                              int c_hi0, const float* mask_weights, const int32_t* pos_hw, int n, int n_pairs, int n_max,
                              void* crop16, float* rs, void* px16, void* stream) {
  if (n == 0) return MASIC_OK;
  const long total = (long)n_pairs * n * (25 * (m / 8) + cin / 8);
  wave_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(ypad16), h16, w16, m / 8, static_cast<const uint4*>(gmm_in16), cin / 8, c_lo / 8,
      c_hi0 / 8, mask_weights, reinterpret_cast<const int2*>(pos_hw), n, n_pairs, n_max, static_cast<uint4*>(crop16),
      rs, static_cast<uint4*>(px16));
  return (int)cudaGetLastError();
}

extern "C" int masic_wave_gather(const void* ypad16, int w16, int m, const void* gmm_in16, int cin, int c_lo, int c_hi0,
                                 const float* mask_weights, const int32_t* pos_hw, int n, void* crop16, float* rs,
                                 void* px16, void* stream) {
  if (!ypad16 || !gmm_in16 || !pos_hw || !crop16 || !px16 || n < 0 || (m % 8) || (cin % 8) || (c_lo % 8) || (c_hi0 % 8))
    return MASIC_EINVAL;
  return launch_wave_gather(ypad16, 0, w16, m, gmm_in16, cin, c_lo, c_hi0, mask_weights, pos_hw, n, 1, n, crop16, rs,
                            px16, stream);
}

extern "C" int masic_wave_gather_pairs(const void* ypad16, int h16, int w16, int m, const void* gmm_in16, int cin,
                                       int c_lo, int c_hi0, const float* mask_weights, const int32_t* pos_hw, int n,
                                       int n_pairs, int n_max, void* crop16, float* rs, void* px16, void* stream) {
  if (!ypad16 || !gmm_in16 || !pos_hw || !crop16 || !px16 || (rs && !mask_weights) || h16 <= 0 || w16 <= 0 || m <= 0 ||
      cin <= 0 || n < 0 || n_pairs <= 0 || n_max < n || (m % 8) || (cin % 8) || (c_lo % 8) || (c_hi0 % 8))
    return MASIC_EINVAL;
  return launch_wave_gather(ypad16, h16, w16, m, gmm_in16, cin, c_lo, c_hi0, mask_weights, pos_hw, n, n_pairs, n_max,
                            crop16, rs, px16, stream);
}

extern "C" int masic_wave_center(const void* ctx_out16, int cin, int c0, int nc, int n, void* px16, void* stream) {
  if (!ctx_out16 || !px16 || n < 0 || (cin % 8) || (c0 % 8) || (nc % 8)) return MASIC_EINVAL;
  if (n == 0) return MASIC_OK;
  const long total = (long)n * (nc / 8);
  wave_center_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(ctx_out16), cin / 8, c0 / 8, nc / 8, n, static_cast<uint4*>(px16));
  return (int)cudaGetLastError();
}

extern "C" int masic_range_streams_init(const uint8_t* data, const int64_t* offsets, int n_streams, void* state,
                                        void* stream) {
  if (!data || !offsets || !state || n_streams <= 0) return MASIC_EINVAL;
  range_streams_init_kernel<<<(n_streams + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      data, offsets, n_streams, static_cast<StreamState*>(state));
  return (int)cudaGetLastError();
}

static int launch_range_decode_wave(const int32_t* rows, int n, int n_streams, int row_pitch, void* state,
                                    const uint8_t* data, const int64_t* offsets, const int32_t* ch_list, int minmax,
                                    const int32_t* s_pair, const int32_t* s_minmax, const int32_t* pos_hw, int h16,
                                    int w16, int m, float* y_nhwc, void* ypad16, int f16, int* error_flag, void* stream) {
  if (n == 0 || n_streams == 0) return MASIC_OK;
  range_decode_wave_kernel<<<(n_streams + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      rows, n, n_streams, row_pitch, static_cast<StreamState*>(state), data, offsets, ch_list, minmax, s_pair, s_minmax,
      reinterpret_cast<const int2*>(pos_hw), h16, w16, m, y_nhwc, static_cast<uint16_t*>(ypad16), f16, error_flag);
  return (int)cudaGetLastError();
}

extern "C" int masic_range_decode_wave(const int32_t* rows, int n, int n_ch, int row_len, void* state, const uint8_t* data,
                                       const int64_t* offsets, const int32_t* ch_list, int minmax, const int32_t* pos_hw,
                                       int w16, int m, float* y_nhwc, void* ypad16, int f16, int* error_flag,
                                       void* stream) {
  if (!rows || !state || !data || !offsets || !ch_list || !pos_hw || !y_nhwc || !ypad16 || !error_flag || n < 0 ||
      n_ch <= 0 || row_len < 2)
    return MASIC_EINVAL;
  return launch_range_decode_wave(rows, n, n_ch, row_len, state, data, offsets, ch_list, minmax, nullptr, nullptr,
                                  pos_hw, 0, w16, m, y_nhwc, ypad16, f16, error_flag, stream);
}

extern "C" int masic_range_decode_wave_pairs(const int32_t* rows, int n, int n_streams, int row_pitch, void* state,
                                             const uint8_t* data, const int64_t* offsets, const int32_t* stream_pair,
                                             const int32_t* stream_ch, const int32_t* stream_minmax, int max_minmax,
                                             const int32_t* pos_hw, int h16, int w16, int m, float* y_nhwc,
                                             void* ypad16, int f16, int* error_flag, void* stream) {
  if (!rows || !state || !data || !offsets || !stream_pair || !stream_ch || !stream_minmax || !pos_hw || !y_nhwc ||
      !ypad16 || !error_flag || n < 0 || n_streams < 0 || max_minmax < 1 || row_pitch < 2 * max_minmax + 2 || h16 <= 0 ||
      w16 <= 0 || m <= 0)
    return MASIC_EINVAL;
  return launch_range_decode_wave(rows, n, n_streams, row_pitch, state, data, offsets, stream_ch, 0, stream_pair,
                                  stream_minmax, pos_hw, h16, w16, m, y_nhwc, ypad16, f16, error_flag, stream);
}

extern "C" int masic_range_encode_streams(const int32_t* intervals, const int64_t* base, const int64_t* stride,
                                          int64_t n_pos, int n_streams, uint8_t* slots, int64_t slot_cap, int64_t* lens,
                                          int* error_flag, void* stream) {
  if (!intervals || !base || !stride || !slots || !lens || !error_flag || n_pos < 0 || n_streams < 0 ||
      slot_cap < 3 * n_pos + 16)
    return MASIC_EINVAL;
  if (n_streams == 0) return MASIC_OK;
  range_encode_streams_kernel<<<(n_streams + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      intervals, base, stride, n_pos, n_streams, slots, slot_cap, lens, error_flag);
  return (int)cudaGetLastError();
}

extern "C" int masic_pack_streams(const uint8_t* slots, int64_t slot_cap, const int64_t* lens, int n_streams,
                                  int64_t* offsets, uint8_t* packed, void* stream) {
  if (!slots || !lens || !offsets || !packed || slot_cap <= 0 || n_streams < 0) return MASIC_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  stream_offsets_kernel<<<1, 1024, 0, st>>>(lens, n_streams, offsets);
  if (n_streams > 0) pack_streams_kernel<<<n_streams, 256, 0, st>>>(slots, slot_cap, offsets, packed);
  return (int)cudaGetLastError();
}

// One range-coded stream per channel: intervals_host is (n_pos, n_ch, 3) int32 in coding order; stream c codes
// intervals_host[:, c, :].  out_host receives the streams back to back, lens_host[c] their byte counts.  HOST buffers.
extern "C" int masic_range_encode_channels(const int32_t* intervals_host, int64_t n_pos, int n_ch, uint8_t* out_host,
                                           int64_t out_cap, int64_t* lens_host) {
  if ((!intervals_host && n_pos > 0) || !out_host || !lens_host || n_pos < 0 || n_ch <= 0) return MASIC_EINVAL;
  std::vector<Enc> encs(static_cast<size_t>(n_ch));
  std::vector<int> bad(static_cast<size_t>(n_ch), 0);
  unsigned hw = std::thread::hardware_concurrency();
  const int n_thr = static_cast<int>(hw ? (hw > 16 ? 16 : hw) : 4);
  auto work = [&](int t) {
    for (int c = t; c < n_ch; c += n_thr) {
      Enc& e = encs[c];
      e.out.reserve(static_cast<size_t>(n_pos) + 16);
      for (int64_t i = 0; i < n_pos; ++i) {
        const int32_t* iv = intervals_host + (i * n_ch + c) * 3;
        if (iv[0] < 0 || iv[1] <= 0 || iv[2] <= 0 || iv[0] + iv[1] > iv[2] || iv[2] > (1 << 22)) { bad[c] = 1; break; }
        e.encode(static_cast<uint32_t>(iv[0]), static_cast<uint32_t>(iv[1]), static_cast<uint32_t>(iv[2]));
      }
      e.finish();
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_thr; ++t) th.emplace_back(work, t);
  work(0);
  for (auto& x : th) x.join();
  int64_t off = 0;
  for (int c = 0; c < n_ch; ++c) {
    if (bad[c]) return MASIC_EINVAL;
    const int64_t len = static_cast<int64_t>(encs[c].out.size());
    if (off + len > out_cap) return MASIC_EINVAL;
    for (int64_t i = 0; i < len; ++i) out_host[off + i] = encs[c].out[static_cast<size_t>(i)];
    lens_host[c] = len;
    off += len;
  }
  return MASIC_OK;
}
