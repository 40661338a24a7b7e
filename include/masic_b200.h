/*
 * masic_b200.h — C ABI of libmasic_b200.so (CUDA, sm_100a only).
 *
 * The reference (ywz978020607/MASIC, a CompressAI fork) has no FFI for this
 * path: every hot op is a stock ATen call reached through nn.Module.forward.
 * Each entry point below therefore names the reference Python call site it
 * replaces (file:line relative to the reference root) instead of an existing
 * binding.  INTEGRATION.md shows the ctypes stub a maintainer of the reference
 * would add to route those call sites here.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; all pointers are DEVICE pointers
 *     unless the parameter name ends in _host;
 *   - every function returns 0 on success, a negative MASIC_E* code on a
 *     rejected argument, or a positive cudaError_t;  no exceptions cross the ABI;
 *   - the caller owns every buffer; `stream` is a cudaStream_t passed as void*;
 *   - no hidden global state except the lazily resolved driver entry point for
 *     cuTensorMapEncodeTiled and per-function cudaFuncSetAttribute calls.
 *
 * Activation layout inside the library ("NHWC-bf16"): [N][H][W][Cpitch] with
 * bfloat16 elements, Cpitch a multiple of 8 (16-byte rows for TMA).  The
 * entropy/warp kernels take the reference's own NCHW fp32 tensors.
 */
#ifndef MASIC_B200_H
#define MASIC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MASIC_IMG_XOFF 2    /* first real pixel column of a padded image row (MASIC_CONV_XFOLD4 input) */
#define MASIC_IMG_XPAD 8    /* extra columns per padded image row                                         */
#define MASIC_FMT_BF16 0    /* 16-bit activation / operand formats: every entry point that reads or writes 16-bit     */
#define MASIC_FMT_F16 1     /* NHWC buffers takes `int f16` = one of these (see csrc/cvt16.cuh for which and why)     */
#define MASIC_FMT_SPLIT 2   /* or-ed in (image producers only): pixels of c <= 4 channels are written as [hi(c) | lo(c)], */
                            /* lo = x - float(hi); MASIC_CONV_XFOLD8 weights repeat for channels c..2c-1 (g_a_conv1)      */
#define MASIC_OK 0
#define MASIC_EINVAL (-1)   /* bad argument (shape, alignment, enum)        */
#define MASIC_ENOSUP (-2)   /* valid request this build does not implement  */
#define MASIC_EDRIVER (-3)  /* cuTensorMapEncodeTiled unavailable / failed  */

/* ---------------------------------------------------------------- version */
int masic_abi_version(void);                 /* bumps on any signature change (2: residual inputs, 3: grouped launches of MasicConvDesc, 4: pack batches, 5: cta_pairs, 6: MASIC_CONV_XFOLD8, 7: masic_rans_*, udh front-end entry points, 8: `int f16` format selectors / MasicConvDesc.f16, 9: in_row_pixels / out_blk_images, 10: masic_warp_perspective_fwd3, 11: one masic_warp_perspective_fwd (fwd2/fwd3 folded in)) */
const char* masic_build_info(void);          /* "sm_100a nvcc 12.9 ..." */

/* ------------------------------------------------------------------ convs */
/* activation fused after bias (reference: nn.ReLU / nn.LeakyReLU(0.01) that
 * follow conv()/deconv() in MASIC.py:173-183, 338-376, 410-444, 678-691)    */
enum { MASIC_ACT_NONE = 0, MASIC_ACT_RELU = 1, MASIC_ACT_LEAKY = 2 };
/* GDN fused into the conv epilogue (reference: compressai/layers/gdn.py:77-92) */
enum { MASIC_GDN_NONE = 0, MASIC_GDN_FWD = 1, MASIC_GDN_INV = 2 };
/* what the implicit GEMM computes */
enum {
  MASIC_CONV = 0,          /* nn.Conv2d(k, stride s, pad k/2)  — models/utils.py:128-135  */
  MASIC_DECONV_S2 = 1,     /* nn.ConvTranspose2d(5, s=2, p=2, op=1) — models/utils.py:138-146 */
  MASIC_DECONV_S2_SUBPIX = 2,/* same op, all 4 output phases stacked on N (for tiny Cout):
                                out buffer is [N][H][W][4*Cout padded], phase-major   */
  MASIC_CONV_XFOLD4 = 3,     /* nn.Conv2d(c<=16 -> Cout, k=5, s=2, p=2) with four horizontal taps folded into
                                one K=64 block (g_a_conv1, MASIC.py:513: 10 MMA groups per tile instead
                                of 25).  The input is a plain 16-channel-pitch image stored with a padded
                                row: [N][H][W+8][16] bf16, pixel x at column x+2, pad columns zero
                                (MASIC_IMG_XOFF / MASIC_IMG_XPAD); the TMA tensor map reads OVERLAPPING
                                4-pixel windows (stride 2 pixels) from it, so nothing is replicated in HBM.
                                Pass in_cpitch = 16, c_in = 64, w_in = the real width W.               */
  MASIC_CONV_XFOLD8 = 4      /* the same layer on an 8-channel-pitch image ([N][H][W+8][8] bf16, same padding): the
                                tensor map reads overlapping 8-PIXEL windows (stride 2 pixels), so all five
                                horizontal taps of a kernel row sit in one K=64 block (K index = pixel * 8 +
                                channel, 48 of 64 used): 5 weight k-blocks and 15 K=16 MMAs per tile instead of 10
                                and 25, half the image bytes.  c <= 8; pass in_cpitch = 8, c_in = 64.       */
};

typedef struct MasicConvDesc {
  int kind;            /* MASIC_CONV | MASIC_DECONV_S2 | MASIC_DECONV_S2_SUBPIX          */
  int ksize;           /* 1, 3 or 5 (square)                                            */
  int stride;          /* 1 or 2 (MASIC_CONV only; deconv kinds are stride 2)           */
  uint32_t tap_mask;   /* bit (ky*ksize+kx) set = live tap; 0 means "all taps".
                          MaskedConv2d mask 'A' (layers.py:68-73) = rows 0,1 + (2,0),(2,1) */
  int n, h_in, w_in;   /* batch and INPUT spatial size                                   */
  int c_in;            /* input channels consumed (multiple of 16)                       */
  int c_out;           /* real output channels                                           */
  int c_out_pad;       /* rows per k-block in the packed weights (multiple of n_tile)    */
  int n_tile;          /* accumulator width: multiple of 16, <= 256                      */
  /* input activation buffer, NHWC bf16 */
  const void* in; int in_cpitch; int in_coff;   /* channel pitch / first channel read    */
  /* packed weights from masic_pack_conv_weights(), bf16 [kblocks][c_out_pad][64]        */
  const void* w_packed;
  const float* bias;   /* [c_out_pad] fp32 or NULL                                       */
  /* output buffer NHWC, bf16 or fp32, written at channel offset out_coff               */
  void* out; int out_cpitch; int out_coff; int out_fp32;
  /* per n-tile activation (MASIC_ACT_*), act[i] applies to channels [i*n_tile,(i+1)*n_tile) */
  uint8_t act[32];
  /* fused GDN: requires c_out == n_tile == 128.  gamma_packed: bf16 [128][128] = gamma'
   * (re-parametrised, gdn.py:80-83), beta: fp32 [128] = beta'                           */
  int gdn; const void* gamma_packed; const float* beta;
  /* optional per-pixel multiplier applied last (mask-weighted fusion, MASIC.py:827):
   * out *= rowscale[((n*H+y)*W+x)*rs_stride + rs_off]                                   */
  const float* rowscale; int rs_stride; int rs_off;
  /* optional residual inputs added after the activation (MASIC_CONV, stride 1 only): NHWC bf16 with the output's
   * spatial size; out = act(conv + bias) * rowscale + residual0 [+ residual1]   (ResidualBlock, layers.py:160-190;
   * Enhancement_Block, MASIC.py:149-164).  Channel c of the output reads residual[... * cpitch + coff + c]. */
  const void* residual0; int res0_cpitch; int res0_coff;
  const void* residual1; int res1_cpitch; int res1_coff;
  /* optional GROUPED launch (block-diagonal weights): several layers that share K = c_in and the spatial size run
   * as one plan, n-tile t of the packed weights reading input channels [in_coff + nt_in_coff[t], +c_in) and writing
   * its n_tile outputs at channel out_coff + nt_out_coff[t] of output image n + nt_out_img[t] (the out buffer then
   * holds out_images >= n images).  HOST arrays of c_out_pad / n_tile ints, copied at plan creation; all three NULL =
   * ordinary convolution.  Used for the three 1x1 entropy-parameter branches (MASIC.py:338-376, :410-444). */
  const int* nt_in_coff; const int* nt_out_coff; const int* nt_out_img; int out_images;
  /* 1: run the plan on CTA PAIRS (clusters of 2, tcgen05.mma.cta_group::2): each CTA stages half of every weight
   * k-block and the pair issues M = 256 MMAs, which cuts the weight traffic per SM.  Pays off on the 128 -> 128 5x5
   * stride-2 layers and the wide 1x1 / 3x3 layers (-3..5 %), not on layers with few tiles or tiny K.
   * Requires n_tile to be a multiple of 32 (each CTA then stages n_tile / 2 rows, a whole number of 16-wide N steps);
   * other n_tile values with cta_pairs = 1 return MASIC_EINVAL. */
  int cta_pairs;
  /* 16-bit format of the input activations, the packed weights, gamma', the residuals and (unless out_fp32) the
   * output: MASIC_FMT_BF16 (training step: gradients need fp32's exponent range) or MASIC_FMT_F16 (inference engines:
   * 11 significant bits instead of 8, same tensor-core rate; conversions saturate at +-65504). */
  int f16;
  /* 1: launch with programmatic stream serialization (PDL): the kernel's prologue (barrier init, TMEM allocation,
   * tensor-map prefetch) overlaps the tail of the previous kernel in the stream, and it lets the NEXT kernel's CTAs be
   * scheduled as soon as SMs free up.  Pays off on chains of tiny launches (the wavefront decoder's per-wave model). */
  int pdl;
  /* MASIC_CONV, stride 1: the input buffer's rows hold in_row_pixels >= w_in pixels (0 = w_in); taps that reach past
   * column w_in read the buffer's own columns instead of zero padding (used with folded-pixel views whose last
   * window hangs over the image edge). */
  int in_row_pixels;
  /* 1: PLANAR output.  The n-tile's 16-channel (fp32) / 32- or 64-channel (16-bit) staging blocks are written to
   * separate output images: block j of image n goes to image n * nblk + j at channel out_coff, i.e. `out` is
   * [n * nblk][H][W][out_cpitch] and channels beyond out_cpitch are clipped.  With out_cpitch = 8 and a pixel-folded
   * input this writes an NCHW fp32 tensor directly (after_conv, MASIC.py:600,616).  Single n-tile plans only. */
  int out_blk_images;
} MasicConvDesc;

typedef struct MasicConvPlan MasicConvPlan;   /* opaque: tensor maps + tile program */

/* Build the TMA tensor maps and the per-tile load/MMA program for one layer.
 * Buffers named in `desc` are bound into the plan (graph-capturable launches). */
int masic_conv_plan_create(const MasicConvDesc* desc, MasicConvPlan** plan_out);
int masic_conv_plan_launch(const MasicConvPlan* plan, void* stream);
void masic_conv_plan_destroy(MasicConvPlan* plan);
/* Training (CQE ResidualBlock backward): a plan with residual0 also stores act(conv + bias), before the residual adds,
 * to channel coff + c of the bf16 NHWC buffer act_out (cpitch, coff multiples of 8; same spatial size as the output).
 * The plan's own output is unchanged.  bf16 plans with a 16-bit output and no rowscale only; MASIC_ENOSUP on CTA
 * pairs, fp16, PDL or planar output.  Plans that never call this launch exactly as before. */
int masic_conv_plan_set_act_out(MasicConvPlan* plan, void* act_out_bf16, int cpitch, int coff);
/* useful work of one launch, for roofline accounting */
int masic_conv_plan_info(const MasicConvPlan* plan, double* flops, double* hbm_bytes,
                         int* n_work_items, int* smem_bytes);

/* Kept for ABI compatibility: the kernels no longer record clock64() stamps, so this always returns
 * MASIC_ENOSUP. */
int masic_conv_plan_trace(const MasicConvPlan* plan, long long* out_host);

/* Pack torch-layout fp32 weights into the bf16 k-block layout the plan reads.
 *   transposed = 0: w is (c_out, c_in, k, k)   [nn.Conv2d]
 *   transposed = 1: w is (c_in, c_out, k, k)   [nn.ConvTranspose2d]
 *   subpix     = 1: build the 3x3 / 4-phase matrix of MASIC_DECONV_S2_SUBPIX
 * dst must hold masic_packed_weight_bytes() bytes.                             */
int64_t masic_packed_weight_bytes(int kind, int ksize, int c_in, int c_out_pad);
int masic_pack_conv_weights(const float* w, int kind, int transposed, int ksize,
                            int c_in, int c_out, int c_out_pad, void* dst, int f16, void* stream);
/* All weight packs of a training step as ONE launch (after every optimizer.step() the kernels' bf16 copies of every
 * conv()/deconv() weight and the padded fp32 biases are refreshed: ~110 packs + ~50 bias copies per step).  A job is
 * one masic_pack_conv_weights() call plus, when bias_src != NULL, bias_dst[i] = bias_src[i % c_out] for
 * i < c_out (4 * c_out for MASIC_DECONV_S2_SUBPIX).  All pointers are DEVICE pointers that stay valid for the life of
 * the batch; the job table itself is host memory, copied at creation. */
typedef struct MasicPackJob {
  const float* w; void* dst; const float* bias_src; float* bias_dst;
  int kind, transposed, ksize, c_in, c_out, c_out_pad;
} MasicPackJob;
typedef struct MasicPackBatch MasicPackBatch;
int masic_pack_batch_create(const MasicPackJob* jobs, int n_jobs, MasicPackBatch** batch_out);
int masic_pack_batch_launch(const MasicPackBatch* batch, void* stream);
void masic_pack_batch_destroy(MasicPackBatch* batch);
/* GDN re-parametrisation (parametrizers.py:61-64) + bf16 pack of gamma:
 *   beta'  = max(beta,  sqrt(beta_min + 2^-36))^2 - 2^-36
 *   gamma' = max(gamma, 2^-18)^2 - 2^-36                                        */
int masic_gdn_prepare(const float* beta, const float* gamma, int c, float beta_min,
                      float* beta_out, float* gamma_out_f32, void* gamma_out_bf16,
                      int f16, void* stream);

/* Plain direct convolution on CUDA cores (test oracle on the device + the
 * small-channel layers).  Same NHWC-bf16 activations, fp32 torch-layout weights. */
int masic_conv_direct_nhwc(const void* in, int n, int h_in, int w_in, int in_cpitch, int in_coff,
                           int c_in, const float* w, int transposed, int ksize, int stride,
                           uint32_t tap_mask, const float* bias, int c_out,
                           float* out_f32, int out_cpitch, int out_coff, int round_w_bf16,
                           int f16, void* stream);


/* --------------------------------------------------------- entropy models */
/* Tensor layouts: `*_nhwc` flags select [N][P][C] (the engine's buffers) instead of the
 * reference's [N][C][P]; P = H*W.  Every output pointer may be NULL (not produced). */

/* GaussianMixtureConditional_gf.forward (compressai/entropy_models/entropy_models.py:808-858;
 * instantiated as HSIC.gaussian1/2, MASIC.py:658-659; called :767,:829):
 *   y_hat = round(y);  lik = max(sum_k w_k [Phi((.5-|y_hat-mu_k|)/s_k) - Phi((-.5-|y_hat-mu_k|)/s_k)], 1e-9)
 *   s_k = max(sigma_k, scale_bound);  parameters are k-major along channels (ch = k*M + m).
 * weights_are_logits=1 fuses the softmax over K of MASIC.py:389-393 / :459-464.
 * yq_bf16 (optional): NHWC bf16 copy of y_hat at channel offset bf_coff of a bf_pitch-wide
 * buffer, times rowscale[(n*P+p)*rs_stride+rs_off] when rowscale != NULL (MASIC.py:827). */
int masic_gmm_likelihood_fwd(const float* y, const float* sigma, const float* mu, const float* weights,
                             int weights_are_logits, int in_nhwc, int n, int m, int k, int hw,
                             float scale_bound, float* y_hat, float* lik, int32_t* symbols, int out_nhwc,
                             void* yq_bf16, int bf_pitch, int bf_coff, const float* rowscale,
                             int rs_stride, int rs_off, int f16, void* stream);

/* GaussianConditional.forward + _quantize('symbols') (entropy_models.py:528-554, :112-125),
 * elementwise over `numel` contiguous values; means may be NULL. */
int masic_gc_likelihood_fwd(const float* y, const float* scales, const float* means, int64_t numel,
                            float scale_bound, float* y_hat, float* lik, int32_t* symbols, void* stream);

/* GaussianConditional.build_indexes (entropy_models.py:556-562): bit-exact int32 indexes. */
int masic_gc_build_indexes(const float* scales, int64_t numel, const float* scale_table, int table_len,
                           float scale_bound, int32_t* indexes, void* stream);

/* EntropyBottleneck.forward (eval) + symbols (entropy_models.py:350-411, :420-423).
 * matrices/biases: HOST arrays of 5 DEVICE pointers, factors: 4 — the ParameterLists
 * _matrices/_biases/_factors with filters (3,3,3,3); quantiles: device (C,1,3).
 * zq_bf16 (optional): NHWC bf16 copy of z_hat, pitch bf_pitch (input of h_s). */
int masic_eb_fwd(const float* z, int in_nhwc, int n, int c, int hw, const float* const* matrices,
                 const float* const* biases, const float* const* factors, const float* quantiles,
                 float* z_hat, float* lik, int32_t* symbols, int out_nhwc, void* zq_bf16, int bf_pitch,
                 int f16, void* stream);

/* EntropyModel._quantize (entropy_models.py:98-125): dequantized = round(x-means)+means,
 * symbols = int32(round(x-means)); round half to even. */
int masic_quantize(const float* x, const float* means, int64_t numel, float* dequantized,
                   int32_t* symbols, void* stream);

/* |y| and round(y) as bf16 NHWC copies of an fp32 NHWC latent (inputs of encode_hyper
 * MASIC.py:184-187, context_prediction :757, the mask-weighted y1_hat_warp term :827). */
int masic_latent_prep(const float* y_nhwc, int64_t n_pixels, int c, void* y_abs_bf16, int abs_pitch,
                      void* y_round_bf16, int rnd_pitch, int rnd_coff, const float* rowscale,
                      int rs_stride, int rs_off, int f16, void* stream);

/* compressai._CXX.pmf_to_quantized_cdf (compressai/cpp_exts/ops/ops.cpp:40-109), HOST buffers.
 * Returns 1 / 2 for the reference's two std::domain_error cases. cdf_host holds n+1 values. */
int masic_pmf_to_quantized_cdf(const float* pmf_host, int n, int precision, uint32_t* cdf_host);
/* EntropyModel._pmf_to_cdf (entropy_models.py:136-142), HOST buffers; cdf is (rows, max_length+2). */
int masic_pmf_table_to_cdf(const float* pmf_host, int rows, int row_stride, const float* tail_mass_host,
                           const int32_t* pmf_length_host, int max_length, int precision,
                           int32_t* cdf_host);

/* Per-symbol coder model of the y bitstream (HSIC.compress / decompress, MASIC.py:1006-1043 and :1263-1300):
 * for every position p < n_pos and listed channel ch_list[j] the K-mixture pmf on the support
 * s = 0 .. 2*minmax (means shifted by +minmax), clipped to [1/65536, 1], normalised to 65536, rounded and
 * prefix-summed in float32 like the reference's numpy code.  sigma/mu/weights: NHWC fp32 (n_pos, K*m),
 * k-major channels.  rows (optional): (n_pos, n_ch, 2*minmax+2) int32, row[0] = 0.  intervals (optional,
 * needs y_hat_nhwc (n_pos, m)): (n_pos, n_ch, 3) int32 = cdf[sym], cdf[sym+1]-cdf[sym], cdf[-1] for
 * sym = y_hat + minmax.  All device pointers. */
int masic_gmm_symbol_cdfs(const float* sigma_nhwc, const float* mu_nhwc, const float* weights_nhwc,
                          int weights_are_logits, int m, int k, int64_t n_pos, const int32_t* ch_list,
                          int n_ch, int minmax, float scale_bound, const float* y_hat_nhwc, int32_t* rows,
                          int32_t* intervals, void* stream);

/* Range coder standing in for the PyPI `range_coder` package the reference calls at MASIC.py:958,1043,1221
 * (RangeEncoder.encode([symbol], cdf) / RangeDecoder.decode(1, cdf)); HOST buffers.  intervals_host is
 * (n, 3) int32 as produced by masic_gmm_symbol_cdfs.  The byte format is this library's own. */
typedef struct MasicRangeDecoder MasicRangeDecoder;
int masic_range_encode(const int32_t* intervals_host, int64_t n, uint8_t* out_host, int64_t out_cap,
                       int64_t* out_len);
int masic_range_decoder_create(const uint8_t* data_host, int64_t len, MasicRangeDecoder** dec_out);
int masic_range_decode_rows(MasicRangeDecoder* dec, const int32_t* rows_host, int n_rows, int row_len,
                            int32_t* symbols_host);
void masic_range_decoder_destroy(MasicRangeDecoder* dec);

/* --- the y payload as one range-coded stream per (view, non-zero channel): "format 2" of masic_b200/bitstream.py ---
 * Same coder arithmetic as masic_range_encode / masic_range_decode_rows, but the symbols of channel c form their own
 * stream, so a GPU warp per channel can decode a whole wave of positions without leaving the device.
 * masic_range_encode_channels (HOST): intervals_host (n_pos, n_ch, 3) in coding order -> streams back to back. */
int masic_range_encode_channels(const int32_t* intervals_host, int64_t n_pos, int n_ch, uint8_t* out_host,
                                int64_t out_cap, int64_t* lens_host);
/* DEVICE side of the wavefront decoder (MASIC.py:1227-1301): state is n_streams x 16 bytes of device memory, data the
 * streams back to back in device memory, offsets (n_streams + 1) int64 byte offsets in device memory. */
int masic_range_streams_init(const uint8_t* data, const int64_t* offsets, int n_streams, void* state, void* stream);
/* decode one symbol per (position of the wave, stream): rows (n, n_ch, row_len) int32 from masic_gmm_symbol_cdfs;
 * symbol - minmax is written to y_nhwc[(h*w16 + w)*m + ch] (fp32) and to the zero-padded 16-bit copy
 * ypad16[((h+2)*(w16+4) + w+2)*m + ch]; pos_hw: n (h, w) int32 pairs; *error_flag != 0 after a corrupt stream. */
int masic_range_decode_wave(const int32_t* rows, int n, int n_ch, int row_len, void* state, const uint8_t* data,
                            const int64_t* offsets, const int32_t* ch_list, int minmax, const int32_t* pos_hw, int w16,
                            int m, float* y_nhwc, void* ypad16, int f16, int* error_flag, void* stream);
/* inputs of a wave's context conv and parameter nets in one launch: 5x5 crops of ypad16 around every position, the
 * position's mask weights replicated over the crop (rs, right view; NULL otherwise), and channels [0, c_lo) and
 * [c_hi0, cin) of gmm_in16 at the position -> px16 (n, cin). */
int masic_wave_gather(const void* ypad16, int w16, int m, const void* gmm_in16, int cin, int c_lo, int c_hi0,
                      const float* mask_weights, const int32_t* pos_hw, int n, void* crop16, float* rs, void* px16,
                      void* stream);
/* px16[i][c0 : c0+nc] = ctx_out16[i][2][2][c0 : c0+nc] (the centre pixel of every crop's context output) */
int masic_wave_center(const void* ctx_out16, int cin, int c0, int nc, int n, void* px16, void* stream);

/* --- format 2 for several pairs at once (HSIC.compress_batch / decompress_batch in masic_b200/bitstream.py) ---
 * All pairs share H, W and so the wave schedule.  A STREAM is one (pair, view, non-zero channel); the stream tables
 * stream_pair / stream_ch / stream_minmax (device int32, n_streams entries) give its pair index, channel and the pair's
 * minmax (1 <= stream_minmax[s] <= max_minmax).  Pair b's tensors follow pair b-1's in every batched buffer.  A count
 * of zero streams or positions is an empty call; negative counts, NULL pointers and misaligned channel counts return
 * MASIC_EINVAL before any launch.  All pointers are device pointers.
 *
 * masic_gmm_symbol_cdfs for listed streams: element (p, s) reads the parameters and y_hat of position
 * stream_pair[s] * pair_stride + p; rows (optional) are (n_pos, n_streams, row_pitch) int32 with
 * row_pitch >= 2 * max_minmax + 2, of which stream s fills 2 * stream_minmax[s] + 2; intervals (optional) are
 * (n_pos, n_streams, 3). */
int masic_gmm_symbol_cdfs_pairs(const float* sigma_nhwc, const float* mu_nhwc, const float* weights_nhwc,
                                int weights_are_logits, int m, int k, int64_t n_pos, int64_t pair_stride,
                                const int32_t* stream_pair, const int32_t* stream_ch, const int32_t* stream_minmax,
                                int n_streams, int max_minmax, float scale_bound, const float* y_hat_nhwc, int32_t* rows,
                                int row_pitch, int32_t* intervals, void* stream);
/* masic_wave_gather for n_pairs pairs: ypad16 (n_pairs, h16+4, w16+4, m), gmm_in16 (n_pairs, h16, w16, cin), mask_weights
 * (n_pairs, h16, w16, 3); position i of pair b goes to row b * n_max + i of crop16 / rs / px16 (n_max >= n). */
int masic_wave_gather_pairs(const void* ypad16, int h16, int w16, int m, const void* gmm_in16, int cin, int c_lo,
                            int c_hi0, const float* mask_weights, const int32_t* pos_hw, int n, int n_pairs, int n_max,
                            void* crop16, float* rs, void* px16, void* stream);
/* masic_range_decode_wave for listed streams: rows (n, n_streams, row_pitch) from masic_gmm_symbol_cdfs_pairs; stream s
 * writes into pair stream_pair[s]'s slice of y_nhwc (n_pairs, h16, w16, m) and ypad16 (n_pairs, h16+4, w16+4, m). */
int masic_range_decode_wave_pairs(const int32_t* rows, int n, int n_streams, int row_pitch, void* state,
                                  const uint8_t* data, const int64_t* offsets, const int32_t* stream_pair,
                                  const int32_t* stream_ch, const int32_t* stream_minmax, int max_minmax,
                                  const int32_t* pos_hw, int h16, int w16, int m, float* y_nhwc, void* ypad16, int f16,
                                  int* error_flag, void* stream);
/* masic_range_encode_channels on the device, one thread per stream: stream s codes the n_pos intervals
 * intervals[(base[s] + i * stride[s]) * 3 + 0..2] (int32 cum, freq, total; base / stride int64) into
 * slots[s * slot_cap ...] (slot_cap >= 3 * n_pos + 16) and writes its byte count to lens[s] (int64).  The bytes equal
 * masic_range_encode_channels' for the same intervals.  *error_flag = 1 after an interval that coder rejects
 * (cum < 0, freq <= 0, cum + freq > total, total > 2^22), 2 after a slot overflow. */
int masic_range_encode_streams(const int32_t* intervals, const int64_t* base, const int64_t* stride, int64_t n_pos,
                               int n_streams, uint8_t* slots, int64_t slot_cap, int64_t* lens, int* error_flag,
                               void* stream);
/* offsets (n_streams + 1) int64 = exclusive prefix sum of lens (offsets[n_streams] = total bytes), then slot s copied
 * to packed[offsets[s] ...]; packed needs room for the total (n_streams * slot_cap always suffices). */
int masic_pack_streams(const uint8_t* slots, int64_t slot_cap, const int64_t* lens, int n_streams, int64_t* offsets,
                       uint8_t* packed, void* stream);

/* rANS serialisation of the z side information with the byte format of the reference's `compressai.ans`
 * extension (compressai/cpp_exts/rans/rans_interface.cpp: BufferedRansEncoder.encode_with_indexes :108-173,
 * flush :175-200, RansDecoder.set_stream :270-276, decode_stream :278-343; reached from
 * EntropyModel.compress / decompress, entropy_models.py:165-239).  The reference hands symbols, indexes and the
 * CDF tables over as Python lists (`.tolist()` of the whole table per call, entropy_models.py:189-194); these
 * entry points take the int32 buffers themselves: cdfs_host is the (n_tables, row_pitch) `_quantized_cdf` tensor,
 * cdf_sizes_host / offsets_host the `_cdf_length` / `_offset` tensors.  HOST buffers; byte strings are identical
 * to the reference extension's for the same inputs (tests/test_rans_cpu.py). */
typedef struct MasicRansEncoder MasicRansEncoder;
typedef struct MasicRansDecoder MasicRansDecoder;
int masic_rans_encoder_create(MasicRansEncoder** enc_out);
int masic_rans_encoder_push(MasicRansEncoder* enc, const int32_t* symbols_host, const int32_t* indexes_host,
                            int64_t n, const int32_t* cdfs_host, int n_tables, int row_pitch,
                            const int32_t* cdf_sizes_host, const int32_t* offsets_host);
/* *data_out points into the encoder and stays valid until the next call on it */
int masic_rans_encoder_flush(MasicRansEncoder* enc, const uint8_t** data_out, int64_t* len_out);
void masic_rans_encoder_destroy(MasicRansEncoder* enc);
int masic_rans_decoder_create(const uint8_t* data_host, int64_t len, MasicRansDecoder** dec_out);
int masic_rans_decoder_decode(MasicRansDecoder* dec, const int32_t* indexes_host, int64_t n,
                              const int32_t* cdfs_host, int n_tables, int row_pitch, const int32_t* cdf_sizes_host,
                              const int32_t* offsets_host, int32_t* symbols_host);
void masic_rans_decoder_destroy(MasicRansDecoder* dec);

/* ------------------------------------------ g_s_conv4: 128 -> 3 transposed conv at image resolution */
/* ConvTranspose2d(128, 3, k=5, s=2, p=2, op=1) (models/utils.py:138-146; MASIC.py:542, :596) in col2im form: one
 * GEMM Z = x W (K = 128, N = 25 taps x 4) on tcgen05 and a shared-memory gather-sum, writing the (n, 3, 2h, 2w) fp32
 * NCHW image directly; gdn = MASIC_GDN_INV additionally applies after_gdn (IGDN over the 3 channels, MASIC.py:599)
 * with the STORED beta (3) / gamma (3x3) given as HOST arrays.  in: NHWC 16-bit, channel pitch 128, h_in % 8 == 0. */
typedef struct MasicDeconvImgPlan MasicDeconvImgPlan;
int64_t masic_deconv_img_weight_bytes(void);
int masic_deconv_img_pack_weights(const float* weight_128x3x5x5, void* dst_16, int f16, void* stream);
int masic_deconv_img_plan_create(const void* in_nhwc16, int n, int h_in, int w_in, int c_pitch, const void* w_packed,
                                 const float* bias3, int gdn, const float* beta3_host, const float* gamma9_host,
                                 float* out_nchw, int f16, MasicDeconvImgPlan** plan_out);
/* Optional second destination of the plan (out_nchw of masic_deconv_img_plan_create may then be NULL): the 3 output
 * channels as 16-bit NHWC at channel coff (even) of pixel slot (y * row_pixels + x + xoff) * c_pitch.  When coff and
 * c_pitch are multiples of 4 the pixel is ONE 8-byte store [c0 c1 c2 0] (channel coff + 3 is zeroed). */
int masic_deconv_img_plan_set_out16(MasicDeconvImgPlan* plan, void* out_nhwc16, int c_pitch, int row_pixels, int xoff,
                                    int coff, int f16);
int masic_deconv_img_plan_launch(const MasicDeconvImgPlan* plan, void* stream);
void masic_deconv_img_plan_destroy(MasicDeconvImgPlan* plan);

/* ---------------------------------------------------- udh homography front-end (SURVEY 8(f)#4) */
/* nn.MaxPool2d(2, 2) of coremasic/mywork/model.py:66 on an NHWC bf16 activation (c_pitch % 8 == 0). */
int masic_maxpool2_nhwc_bf16(const void* in, int n, int h, int w, int c_pitch, void* out, int f16, void* stream);
/* nn.Linear weights (rows, c*hw) whose columns follow torch's Flatten of NCHW (model.py:83-87) -> bf16 (rows, hw*c):
 * the column order of the NHWC activation the FC kernel reads. */
int masic_fc_pack_weights(const float* weight, int rows, int c, int hw, void* dst_bf16, int f16, void* stream);
/* nn.Linear (+ReLU) for batch <= 8 (model.py:87-90): out[b][r] = act(bias[r] + w[r] . x[b]); x, w bf16, fp32
 * accumulation; out as fp32 and / or bf16.  HBM-bound on the weight matrix (read once per call). */
int masic_fc_bf16(const void* x_bf16, int x_batch_stride, const void* w_bf16, const float* bias, int batch, int k,
                  int rows, int relu, float* out_f32, void* out_bf16, int out_batch_stride, int f16, void* stream);
/* test2_real.py:201-211 / model.py:103-111: corners (batch,4,2) and the net's delta (batch,4,2), fp32 ->
 * h_matrix (batch,3,3) fp32 = h_adjust(img_h, img_w, pic_h, pic_w, inverse(get_perspective_transform(c', c' + delta)))
 * with c' = c - c[0] when shift_corners (test2_real.py:203) else c (model.py get_h; img == pic makes h_adjust the
 * identity).  8x8 solve and 3x3 inverse in fp64. */
int masic_homography_from_delta(const float* corners, const float* delta, int batch, int shift_corners, int img_h,
                                int img_w, int pic_h, int pic_w, float* h_out, void* stream);
/* The (n,3,3) fp32 homographies h_in in the zero-padded frame: h_out = T h_in T^-1, T the translation by (left, top)
 * (pixel coordinates, as the warp reads them).  fp64, one thread per matrix, each product and sum rounded in a fixed
 * order, rounded once to fp32.  h_out may be h_in. */
int masic_homography_pad(const float* h_in, int n, int top, int left, float* h_out, void* stream);

/* ------------------------------------------------------------ image domain */
/* kornia.warp_perspective(src, M, (h_out, w_out)) — kornia 0.5.0, call sites MASIC.py:781,821,833.
 * Step 1: T = inv(N_dst M inv(N_src)) per batch element (invert_m=1 first replaces M by
 * inv(M): the second warp of mask(), MASIC.py:644).  t_out is (batch,3,3) fp64 on device. */
int masic_warp_prepare(const float* m_3x3, int batch, int h, int w, int h_out, int w_out, int invert_m,
                       double* t_out, void* stream);
/* Step 2: bilinear, zero padding, align_corners=True.  src NCHW fp32 with c <= 8 channels;
 * src == NULL warps an all-ones image (mask(), MASIC.py:636-638).  Outputs (any may be NULL, not all):
 *   dst_nchw       NCHW fp32;
 *   dst_nhwc_bf16  NHWC 16-bit (format f16) zero-padded to bf_pitch channels, rows as in the layout packs below;
 *   dst2_nhwc16    a second 16-bit NHWC image (plain MASIC_FMT_BF16 / MASIC_FMT_F16 in d2_f16): the c warped channels
 *                  are written at channel d2_coff of pixel slot (y * d2_row_pixels + x + d2_xoff) * d2_pitch, leaving
 *                  the slot's other channels untouched — several producers fill one channels-last image (the input of
 *                  the tensor-core after_conv).  With c = 3 and d2_coff, d2_pitch multiples of 4 the pixel is ONE
 *                  8-byte store [c0 c1 c2 0] (channel d2_coff + 3 is zeroed);
 *   dst_ones_nchw  (n,1,h_out,w_out): the warp of the ALL-ONES image under the same transform (mask(),
 *                  MASIC.py:636-638: x1_mask_R) from the same launch — the coordinates are evaluated once for both. */
int masic_warp_perspective_fwd(const float* src, int n, int c, int h, int w, int h_out, int w_out,
                               const double* t_prepared, float* dst_nchw, void* dst_nhwc_bf16, int bf_pitch,
                               int bf_row_pixels, int bf_xoff, int f16, void* dst2_nhwc16, int d2_pitch,
                               int d2_row_pixels, int d2_xoff, int d2_coff, int d2_f16, float* dst_ones_nchw,
                               void* stream);

/* Direct conv for the tiny-channel layers (c_in <= 8, c_out <= 8) on NCHW fp32:
 *   Encoder2.pre_conv+pre_gdn (MASIC.py:573-574): in0=x1_warp, in1=x2, k=5, s=1, gdn=FWD
 *   Decoder2.after_conv       (MASIC.py:616):     transposed_s1=1 (ConvTranspose2d weight layout)
 *   mask2weights.maskconv     (MASIC.py:475-488): k=3, s=2, ReLU
 * weight is torch layout (c_out, c0+c1, k, k), or (c0+c1, c_out, k, k) when transposed_s1. */
int masic_conv_small_nchw(const float* in0, int c0, const float* in1, int c1, int n, int h, int w,
                          const float* weight, int transposed_s1, const float* bias, int c_out,
                          int ksize, int stride, int act, int gdn, const float* beta,
                          const float* gamma, float beta_min, float* out_nchw, void* out_nhwc_bf16,
                          int bf_pitch, int bf_row_pixels, int bf_xoff, int f16, void* stream);

/* Output of a MASIC_DECONV_S2_SUBPIX plan ([N][H/2][W/2][pitch] fp32, channel = phase*3+co)
 * -> NCHW fp32 image (N,3,H,W), optionally through GDN/IGDN over the 3 channels
 * (Decoder2.after_gdn, MASIC.py:599,615), optionally also NHWC bf16. */
int masic_subpix_to_nchw(const float* in_nhwc, int n, int h2, int w2, int pitch, int gdn,
                         const float* beta, const float* gamma, float beta_min, float* out_nchw,
                         void* out_nhwc_bf16, int bf_pitch, int f16, void* stream);

/* Stand-alone GDN.forward (compressai/layers/gdn.py:77-92) on NCHW fp32, c <= 256; beta/gamma are
 * the STORED (re-parametrised) parameters, the kernel applies parametrizers.py:61-64 itself. */
int masic_gdn_nchw(const float* x, int n, int c, int hw, const float* beta, const float* gamma,
                   float beta_min, int inverse, float* out, void* stream);

/* softmax over the c (<= 8) channels of an NCHW tensor (mask2weights, MASIC.py:497-502). */
int masic_softmax_channels(const float* in_nchw, int n, int c, int hw, float* out_nchw, float* out_nhwc,
                           void* stream);
/* mask2weights.forward (MASIC.py:472-506) in one launch: the four conv3x3 stride-2 layers (1->3 ReLU, 3->6 ReLU, 6->6 ReLU,
 * 6->3; torch weight layouts, biases may be NULL) and the softmax over the 3 outputs.  mask: (n,1,h,w) fp32.  Outputs
 * (either may be NULL): (n,3,h/16,w/16) NCHW and/or [n][h/16][w/16][3] NHWC, sizes rounded up at every level.  Bit-identical
 * to four masic_conv_small_nchw launches + masic_softmax_channels. */
int masic_mask2weights(const float* mask_nchw, int n, int h, int w, const float* w1, const float* b1, const float* w2,
                       const float* b2, const float* w3, const float* b3, const float* w4, const float* b4,
                       float* out_nchw, float* out_nhwc, void* stream);
/* layout packs.  The NHWC bf16 outputs of this function, of masic_warp_perspective_fwd (both 16-bit destinations) and
 * of masic_conv_small_nchw may have a padded row: pixel (y,x) goes to out[(y*row_pixels + x + xoff)*pitch];
 * row_pixels = 0 means a dense image (row_pixels = w, xoff = 0). */
int masic_nchw_to_nhwc_bf16(const float* in_nchw, int n, int c, int h, int w, void* out, int pitch,
                            int row_pixels, int xoff, int f16, void* stream);
int masic_nhwc_to_nchw_f32(const float* in_nhwc, int n, int c, int hw, int in_pitch, float* out_nchw,
                           void* stream);
/* 8-bit image -> float32 in [0,1]: torchvision.transforms.ToTensor as the reference's datasets apply it
 * (img.float().div(255), IEEE division); lets a caller ship 8-bit images over PCIe (PairStream.submit). */
int masic_u8_to_unit_f32(const uint8_t* in_u8, int64_t numel, float* out_f32, void* stream);
/* Zero padding of NCHW images (n,c,h,w) into the float32 frame (n,c,hp,wp), source pixel (y,x) at (y+top, x+left): the
 * codec's frame for pairs whose size is not a multiple of 64 (masic_b200/padding.py).  src is uint8 (src_u8 = 1,
 * converted like masic_u8_to_unit_f32, bit for bit) or float32 (copied).  Every element of dst is written, the zero
 * border included, so dst needs no memset.  dst_unpadded (may be NULL): the float32 (n,c,h,w) image from the same pass.
 * Memory-bound: n*c*(h*w*s_in + hp*wp*4 [+ h*w*4]) bytes; 16-byte stores when wp % 4 == 0 and dst is 16-byte aligned. */
int masic_pad_image(const void* src, int src_u8, int n, int c, int h, int w, int hp, int wp, int top, int left,
                    float* dst, float* dst_unpadded, void* stream);

/* ------------------------------------------------- cross quality enhancement (CQE) glue */
/* Independent_EN (coremasic/mywork/MASIC.py:1436-1501).  Its 3x3 convs run as MASIC_CONV plans with LeakyReLU and
 * the ResidualBlock / Enhancement_Block adds fused (MasicConvDesc.residual0/1); these are the blends around them.
 * weights_nchw2 = softmax output of mask2weights_EN, (N,2,H,W) fp32: channel 0 weighs the OTHER view's warped map,
 * channel 1 this view's own map. */
/* mask2weights_EN.forward (MASIC.py:1411-1434) fused: 4x conv3x3 stride 1 (1->kw->2kw->2kw->kw, ReLU between, each
 * zero-padding its own input) + softmax over the kw channels; mask (N,1,H,W) fp32 -> weights (N,kw,H,W) fp32.
 * weights4 / biases4: HOST arrays of 4 DEVICE pointers in torch Conv2d layout.  kw must be 2. */
int masic_cqe_mask_weights(const float* mask_nchw1, int n, int h, int w, const float* const* weights4,
                           const float* const* biases4, int kw, float* out_nchw2, void* stream);
/* MASIC.py:1470-1471: out[p][0:3] = a[:,p]*w0[p], out[p][3:6] = b[:,p]*w1[p], out[p][6:16] = 0 (NHWC bf16, pitch 16);
 * a = the other view warped (NCHW fp32), b = this view's image. */
int masic_cqe_blend_images(const float* a_nchw, const float* b_nchw, const float* weights_nchw2, int n, int h,
                           int w, void* out_nhwc16_bf16, int f16, void* stream);
/* MASIC.py:1479-1482: out[p][0:c] = self[p]*w1[p]; out[p][c:2c] = warp_perspective(other, M)[p]*w0[p] (bilinear,
 * zeros, align_corners=True; t_prepared from masic_warp_prepare with src = dst = (h, w)).  NHWC bf16, c % 8 == 0. */
int masic_cqe_feature_fuse(const void* self_bf16, int self_pitch, const void* other_bf16, int other_pitch,
                           int c, const float* weights_nchw2, const double* t_prepared, int n, int h, int w,
                           void* out_bf16, int out_pitch, int f16, void* stream);
/* MASIC.py:1495-1496: out_nchw[b][c][p] = conv_out_nhwc[b][p][c] + identity_nchw[b][c][p], c < 3 (fp32). */
int masic_cqe_residual_image(const float* conv_out_nhwc, int pitch, const float* identity_nchw, int n, int h,
                             int w, float* out_nchw, void* stream);
/* Training.  Backward of masic_cqe_feature_fuse for one view, g = dL/d(out) (bf16, pitch g_pitch >= 2c):
 *   d_self[p][0:c] = g[p][0:c] * w1[p]                                      (bf16, written)
 *   d_other += transpose of the bilinear warp of g[p][c:2c] * w0[p]        (fp32 NHWC, atomics: zero it first)
 *   dweights[p][0] = sum_c g[p][c+.] * warp(other)[p][.],  dweights[p][1] = sum_c g[p][.] * self[p][.]
 *                                                                           (NHWC (N,H,W,2) fp32, written)
 * The two views cross: view L's fuse warps EB1(R) by H^-1, so its d_other is EB1(R)'s gradient, and the reverse. */
int masic_cqe_feature_fuse_bwd(const void* g_bf16, int g_pitch, const void* self_bf16, int self_pitch,
                               const void* other_bf16, int other_pitch, int c, const float* weights_nchw2,
                               const double* t_prepared, int n, int h, int w, void* d_self_bf16, int d_self_pitch,
                               float* d_other_f32, int d_other_pitch, float* dweights_nhwc2, void* stream);
/* Backward of masic_cqe_blend_images w.r.t. the weights only (the images come from the frozen codec):
 * dweights[p][0] += sum_c g[p][c] a[c][p], dweights[p][1] += sum_c g[p][3+c] b[c][p]; g fp32 NHWC (pitch >= 6). */
int masic_cqe_blend_images_bwd(const float* g_nhwc, int g_pitch, const float* a_nchw, const float* b_nchw, int n,
                               int h, int w, float* dweights_nhwc2, void* stream);

/* ------------------------------------------------------------- criterion */
/* RateDistortionLoss.forward (coremasic/mywork/test2_real.py:88-114, newtrain_codec_real.py:66-87) on the
 * output of HSIC.forward: out8 (device, 8 floats) = { bpp of the 4 likelihood tensors (y1,y2,z1,z2 or any order),
 * mse view 1, mse view 2, bpp total, lambda*255^2*(mse1+mse2)+bpp }.  bpp_t = sum(log lik_t) / (-ln2 * n*h*w);
 * mse_v = mean over n*c*h*w.  lik4_host / lik_numel4_host are HOST arrays of 4 device pointers / element
 * counts (a NULL pointer skips the tensor); scratch is masic_rd_metrics_scratch_bytes() of device memory.
 * Two launches, deterministic (fixed-order fp64 reduction). */
int64_t masic_rd_metrics_scratch_bytes(void);
int masic_rd_metrics(const float* const* lik4_host, const int64_t* lik_numel4_host, const float* x1_hat,
                     const float* x1, const float* x2_hat, const float* x2, int n, int c, int h, int w,
                     float lmbda, void* scratch, float* out8, void* stream);
/* pytorch_msssim.ms_ssim / ssim (version 1.0) of two NCHW fp32 batches x, y (device), as the reference's eval loop
 * reports it next to bpp and PSNR (coremasic/mywork/test2_real.py:88-114; test3_real.py after the enhancement net):
 * out_nc (device, n*c floats) = per-(n, c) value.  11-tap Gaussian window (sigma 1.5, float32 taps computed on the host
 * as the package does), valid correlation, C1 = (k1*data_range)^2, C2 = (k2*data_range)^2; `levels` (1..5) scales with
 * avg_pool2d(2, padding (h%2, w%2), count_include_pad) between them; value = prod_{l<levels-1} relu(mean cs_l)^w_l
 * * s^w_{levels-1}, s = mean ssim of the last level, relu'd when nonneg_last != 0 (ms_ssim always, ssim with
 * nonnegative_ssim).  levels = 1 with weights {1} is ssim.  weights_host: HOST array of `levels` floats.  Every level
 * must be at least 11 x 11 (MASIC_EINVAL otherwise).  scratch is masic_ms_ssim_scratch_bytes() of device memory (the
 * pyramid and per-tile partial sums).  Deterministic (fixed-order fp64 reduction) and batch invariant: a plane's value
 * does not depend on the other planes of the call. */
int64_t masic_ms_ssim_scratch_bytes(int n, int c, int h, int w, int levels);
int masic_ms_ssim(const float* x, const float* y, int n, int c, int h, int w, int levels, float data_range, float k1,
                  float k2, const float* weights_host, int nonneg_last, void* scratch, float* out_nc, void* stream);
/* Gradient of masic_ms_ssim with respect to its first argument: dx (device, NCHW fp32 like x) =
 * grad_scale * d(sum over the n*c planes of out_nc)/dx [+ addend].  addend (device, or NULL) may be dx itself.
 * fwd_scratch must hold the scratch of a masic_ms_ssim call with the same x, y, sizes and constants, issued earlier on
 * the same stream (or completed before this call) and not overwritten since: the backward reads that call's pyramid
 * levels 1..levels-1 and re-adds its per-tile partial sums in the final launch's order, so the level means it
 * differentiates are the ones behind the forward's value.  A level whose relu'd mean clamps to 0 contributes 0 and, as
 * in torch's prod backward, zeroes the gradient of every other level.  work is masic_ms_ssim_bwd_work_bytes() of device
 * memory (per-level coefficient maps and gradients).  2 + levels launches; deterministic (no atomics) and batch
 * invariant.  MASIC_EINVAL for the sizes masic_ms_ssim rejects and for a NULL x, y, weights_host, fwd_scratch, dx or
 * work. */
int64_t masic_ms_ssim_bwd_work_bytes(int n, int c, int h, int w, int levels);
int masic_ms_ssim_bwd(const float* x, const float* y, int n, int c, int h, int w, int levels, float data_range,
                      float k1, float k2, const float* weights_host, int nonneg_last, const void* fwd_scratch,
                      float grad_scale, const float* addend, float* dx, void* work, void* stream);
/* lpips.LPIPS(net='alex') (lpips 0.1, version '0.1'), as the reference's eval loop reports it next to bpp, PSNR and
 * MS-SSIM (coremasic/mywork/test2_real.py:88-114; test3_real.py).  The five AlexNet convolutions run as conv_tc plans;
 * these four entry points are the rest.  All activations are fp16 NHWC; a batch holds 2n images and image i is
 * compared with image i + n.  Feature maps: ho = (h - 7) / 4 + 1, h2 = (ho - 3) / 2 + 1, h3 = (h2 - 3) / 2 + 1
 * (floor; the same for widths); every entry point that takes (h, w) returns MASIC_EINVAL unless h, w >= 31 (all maps
 * non-empty).
 *
 * masic_lpips_prep replaces `2 * x - 1` (forward(normalize=True)) and ScalingLayer.forward, `(x - shift) / scale`:
 * imgs is a DEVICE array of n device pointers to (3, h, w) fp32 images; out = [n][ho + 2][wo + 2][64] fp16 4x4
 * space-to-depth blocks: channel (r * 4 + s) * 3 + ch of block (bi, bj) = the scaled pixel (4 bi - 2 + r, 4 bj - 2 + s)
 * of channel ch rounded to fp16 (zero outside the image, channels 48..63 zero).  AlexNet's conv1 (11x11, stride 4,
 * pad 2) is then a 3x3 stride-1 conv over 48 channels (weights folded by masic_b200.convplan.fold_s2d4_weights_11x11)
 * whose "same" output at (i + 1, j + 1) is conv1's output (i, j).  shift_host / scale_host: HOST arrays of 3 floats. */
int masic_lpips_prep(const float* const* imgs, int n, int h, int w, int normalize, const float* shift_host,
                     const float* scale_host, void* out, void* stream);
/* torch.nn.MaxPool2d(3, stride 2) (AlexNet features[2], [5]; floor mode, no padding) of the h x w window at
 * (y0, x0) of an [n][in_rows][in_cols][c] fp16 buffer (the origin lets it read relu1 inside conv1's output on the
 * space-to-depth grid) -> out [n][(h - 3) / 2 + 1][(w - 3) / 2 + 1][c].  c a multiple of 8, h, w >= 3. */
int masic_maxpool3s2_nhwc(const void* in, int n, int in_rows, int in_cols, int y0, int x0, int h, int w, int c,
                          void* out, void* stream);
/* LPIPS.forward's head: per layer k, normalize_tensor (f / (sqrt(sum_c f^2) + 1e-10)) of both features, the squared
 * difference, the 1x1 lin{k} conv (no bias) and spatial_average; then the sum over the layers.  feat_host: HOST array
 * of 5 device pointers, [2n][ho + 2][wo + 2][64] (conv1's output, relu1 at origin (1, 1)), [2n][h2][w2][192],
 * [2n][h3][w3][384], [2n][h3][w3][256] x 2; lin_host: HOST array of 5 device pointers to 64 / 192 / 384 / 256 / 256
 * fp32 weights.  out_layers (device, n * 5 floats) = the per-layer values (retPerLayer), out_total (device, n floats)
 * = their sum.  scratch is masic_lpips_distance_scratch_bytes() of device memory (one fp64 partial sum per
 * 128-pixel block).  Deterministic (fixed-order fp64 reduction) and batch invariant. */
int64_t masic_lpips_distance_scratch_bytes(int n, int h, int w);
int masic_lpips_distance(const void* const* feat_host, const float* const* lin_host, int n, int h, int w,
                         void* scratch, float* out_layers, float* out_total, void* stream);

/* ------------------------------------------------------- training: weight gradients */
/* dW[cl][ch][ky][kx] = sum_{n,p} LO[n,p,cl] * HI[n, stride*p + k - ksize/2, ch]  on the tensor cores
 * (reference: loss.backward() of newtrain_codec_real.py:134 -> ATen convolution_backward for every
 * conv()/deconv() of compressai/models/utils.py:128-146).
 *   nn.Conv2d          (W = (Cout,Cin,k,k)):  LO = dL/d(output), HI = layer input
 *   nn.ConvTranspose2d (W = (Cin,Cout,k,k)):  LO = layer input,  HI = dL/d(output)
 * LO is [n][h_lo][w_lo][lo_cpitch], HI is [n][stride*h_lo][stride*w_lo][hi_cpitch], both NHWC bf16; c_lo, c_hi
 * >= 16 are the real channel counts (the kernel reads whole 64/128-channel tiles: what lies beyond the real
 * count, in the buffer or zero-filled outside it, only reaches rows/columns that are never written to dW).  dw is fp32 in the torch layout of the layer's weight; accumulate=1 adds to it (a layer that runs
 * twice per step, encoder1: MASIC.py:746,822).  Deterministic (fixed-order partial sums in `workspace`). */
typedef struct MasicWgradDesc {
  int ksize, stride;          /* 1/3/5, 1/2 */
  uint32_t tap_mask;          /* as MasicConvDesc.tap_mask; masked taps are left untouched in dw */
  int n, h_lo, w_lo;
  const void* lo; int lo_cpitch, lo_coff, c_lo;
  const void* hi; int hi_cpitch, hi_coff, c_hi;
  float* dw;
  int accumulate;
} MasicWgradDesc;
typedef struct MasicWgradPlan MasicWgradPlan;
int masic_wgrad_plan_create(const MasicWgradDesc* desc, MasicWgradPlan** plan_out);
int64_t masic_wgrad_plan_workspace_bytes(const MasicWgradPlan* plan);
int masic_wgrad_plan_launch(const MasicWgradPlan* plan, void* workspace, void* stream);
int masic_wgrad_plan_info(const MasicWgradPlan* plan, double* flops, int* n_ctas);
void masic_wgrad_plan_destroy(MasicWgradPlan* plan);

/* 3-channel side of g_a_conv1 (Conv2d 3->128) / g_s_conv4 (ConvTranspose2d 128->3), k = 5, stride 2 (CUDA cores):
 * dw[cl][ci][ky][kx] += sum LO[n,p,cl] * HI[n][ci][2p + k - 2];  LO NHWC bf16 [n][h_lo][w_lo][lo_pitch],
 * HI NCHW fp32 [n][c_hi<=4][2 h_lo][2 w_lo].  Accumulates (atomics) into dw. */
int masic_wgrad_small(const void* lo_bf16, int lo_pitch, int c_lo, const float* hi_nchw, int c_hi, int n,
                      int h_lo, int w_lo, float* dw_accum, void* stream);

/* --------------------------------------------- training: entropy models (forward + local backward) */
/* GaussianMixtureConditional_gf.forward in train() mode (entropy_models.py:808-858, 'noise' quantisation :103-110)
 * fused with the backward of the rate term  lik_grad_scale * sum(log lik),  lik_grad_scale = -1/(ln2 * N*H*W)
 * (newtrain_codec_real.py:73-76).  All tensors NHWC: y/noise/lik/y_hat/dy [n_pixels][m]; sigma (post-ReLU), mu,
 * wlogits and the bf16 gradients [n_pixels][k*m], k-major.  dsigma already includes the final ReLU of the sigma
 * branch and the LowerBound(0.11) gradient rule (bound_ops.py:40-42); dwl is w.r.t. the logits (softmax fused). */
int masic_gmm_likelihood_train(const float* y, const float* noise, const float* sigma, const float* mu,
                               const float* wlogits, int64_t n_pixels, int m, int k, float scale_bound,
                               float lik_grad_scale, float* lik, void* y_hat_bf16, int bf_pitch, float* y_hat,
                               float* dy, void* dsigma_bf16, void* dmu_bf16, void* dwl_bf16, void* stream);
/* EntropyBottleneck.forward in train() mode (entropy_models.py:384-411) + backward of its rate term.
 * z/noise/dz NHWC fp32 [n*hw][c]; z_hat/lik NCHW fp32; zq NHWC bf16.  dparams [c][58] = gradients w.r.t. the RAW
 * parameters, per channel: matrices 0..4 (3,9,9,9,3 values, row-major (out,in)), biases 0..4 (3,3,3,3,1),
 * factors 0..3 (3 each). */
int masic_eb_train(const float* z_nhwc, const float* noise_nhwc, int n, int c, int hw,
                   const float* const* matrices, const float* const* biases, const float* const* factors,
                   float lik_grad_scale, float* z_hat_nchw, float* lik_nchw, void* zq_bf16, int bf_pitch,
                   float* dz_nhwc, float* dparams, void* stream);
/* EntropyBottleneck.loss (entropy_models.py:345-348): *loss += sum |logits(quantiles) - target|, dquantiles (c,1,3). */
int masic_eb_aux_loss(const float* quantiles, int c, const float* const* matrices, const float* const* biases,
                      const float* const* factors, const float* target3_host, float* loss, float* dquantiles,
                      void* stream);

/* ------------------------------------- training: element-wise backward over NHWC bf16 [pixels][pitch] */
/* g *= act'(y) in place (ReLU / LeakyReLU(0.01) after conv()/deconv()); bias_grad[c] += sum_p g (may be NULL). */
int masic_act_bwd_bias(void* g_bf16, int g_pitch, int g_coff, const void* y_bf16, int y_pitch, int y_coff,
                       int act, int64_t n_pixels, int c, float* bias_grad, void* stream);
/* The same out of place: dst = g * act'(y), g unchanged (a residual block's skip still reads it). */
int masic_act_bwd_bias_out(const void* g_bf16, int g_pitch, int g_coff, const void* y_bf16, int y_pitch, int y_coff,
                           int act, int64_t n_pixels, int c, void* dst_bf16, int dst_pitch, int dst_coff,
                           float* bias_grad, void* stream);
/* GDN.forward as separate steps (gdn.py:77-92) keeping x and norm for the backward: sq = x^2; (norm = 1x1 conv on
 * the tensor cores); y = x * rsqrt(norm) (inverse: x * sqrt(norm)). */
int masic_gdn_square(const void* x_bf16, void* sq_bf16, int64_t numel, void* stream);
int masic_gdn_apply(const void* x_bf16, const float* norm, int inverse, void* y_bf16, int64_t numel, void* stream);
/* GDN backward: (a) t = dL/dnorm, written to t_bf16; g := g * norm^(-+1/2) in place; dbeta'[c] += sum_p t.
 * (b) after v = gamma'^T t (1x1 conv): u := u + 2 x v in place (= dL/dx); dbias[c] += sum_p (may be NULL). */
int masic_gdn_bwd_a(void* g_bf16, const void* x_bf16, const float* norm, int inverse, void* t_bf16,
                    int64_t n_pixels, int c, float* dbeta_prime, void* stream);
int masic_gdn_bwd_b(void* u_bf16, const void* x_bf16, const float* v, int64_t n_pixels, int c, float* dbias,
                    void* stream);
/* NonNegativeParametrizer backward with LowerBound's rule (parametrizers.py:61-64, bound_ops.py:40-42). */
int masic_reparam_bwd(const float* dprime, const float* stored, int n, float minimum, int accumulate,
                      float* dstored, void* stream);
/* All reparam backwards of a training step as ONE launch (15 GDN layers x {beta, gamma}): HOST arrays of n_jobs device
 * pointers / sizes / minima / accumulate flags (NULL = 0), copied at creation. */
typedef struct MasicReparamBatch MasicReparamBatch;
int masic_reparam_batch_create(const float* const* dprime, const float* const* stored, float* const* dstored,
                               const int* numel, const float* minimum, const int* accumulate, int n_jobs,
                               MasicReparamBatch** out);
int masic_reparam_batch_launch(const MasicReparamBatch* batch, void* stream);
void masic_reparam_batch_destroy(MasicReparamBatch* batch);
int masic_latent_prep_train(const float* y_nhwc, const float* noise_nhwc, int64_t n_pixels, int c,
                            void* y_abs_bf16, int abs_pitch, void* y_noisy_bf16, int noisy_pitch, void* stream);
/* dy = dy_lik + d_dec + d_ctx + sign(y) * d_abs (NULL sources are skipped) -> bf16 */
int masic_latent_merge_bwd(const float* y_nhwc, const float* dy_lik, const void* d_dec_bf16, const void* d_ctx_bf16,
                           const void* d_abs_bf16, int64_t numel, void* dy_bf16, void* stream);
int masic_add_f32_bf16(const float* a, const void* b_bf16, int64_t numel, void* out_bf16, void* stream);
/* cat(params2*w0, ctx2*w1, (y1w+noise)*w2) (MASIC.py:827) and its backward; mask weights NHWC [pixels][3]. */
int masic_mask_fuse_fwd(const void* p2_bf16, const void* c2_bf16, int c2, const float* y1w_nhwc,
                        const float* noise_nhwc, int m, const float* mask_weights_nhwc, int64_t n_pixels,
                        void* fused_bf16, void* stream);
int masic_mask_fuse_bwd(const void* g_bf16, const void* p2_bf16, const void* c2_bf16, int c2, const float* y1w_nhwc,
                        const float* noise_nhwc, int m, const float* mask_weights_nhwc, int64_t n_pixels,
                        void* dp2_bf16, void* dc2_bf16, void* dy1w_bf16, float* dmask_weights_nhwc, void* stream);

/* --------------------------------------------------- training: image domain (NCHW fp32, <= 8 channels) */
/* g = scale * (x_hat - x) [+ addend]: nn.MSELoss backward (newtrain_codec_real.py:78-79). */
int masic_mse_grad(const float* x_hat, const float* x, const float* addend, float scale, int64_t numel, float* g,
                   void* stream);
/* kornia.warp_perspective backward w.r.t. src (g = g0 [+ g1]); dsrc must be zeroed by the caller (atomics). */
int masic_warp_perspective_bwd(const float* g0, const float* g1, int n, int c, int h, int w, int h_out, int w_out,
                               const double* t_prepared, float* dsrc_zeroed, void* stream);
/* backward of masic_conv_small_nchw: g_out is dL/d(output); act_out != NULL masks it with (act_out > 0) (ReLU);
 * din0/din1 (optional) receive dL/d(inputs); dweight/dbias (optional, zeroed by the caller) accumulate. */
int masic_conv_small_bwd(const float* in0, int c0, const float* in1, int c1, int n, int h, int w,
                         const float* weight, int transposed_s1, int c_out, int ksize, int stride,
                         const float* g_out, const float* act_out, float* din0, float* din1,
                         float* dweight_zeroed, float* dbias_zeroed, void* stream);
/* backward of masic_gdn_nchw: dx, and the gradients of beta' / gamma' (accumulated; chain with masic_reparam_bwd). */
int masic_gdn_small_bwd(const float* x, const float* g, int n, int c, int hw, const float* beta,
                        const float* gamma, float beta_min, int inverse, float* dx, float* dbeta_prime_zeroed,
                        float* dgamma_prime_zeroed, void* stream);
int masic_softmax_channels_bwd(const float* w_nhwc, const float* dw_nhwc, int n, int c, int hw,
                               float* dlogits_nchw, void* stream);
int masic_colsum_nchw(const float* g, int n, int c, int64_t hw, float* out_accum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MASIC_B200_H */
