// conv_tc.cu — implicit-GEMM convolution / transposed convolution on the 5th-gen tensor
// cores (tcgen05.mma, accumulators in TMEM), operands staged by TMA, GDN/IGDN fused
// into the epilogue.  sm_100a only.
//
// Replaces (reference, file:line):
//   conv()/deconv() factories          compressai/models/utils.py:128-146
//   GDN.forward                        compressai/layers/gdn.py:77-92
//   MaskedConv2d.forward               compressai/layers/layers.py:75-78
//   the nn.ReLU / nn.LeakyReLU that follow them in MASIC.py:173-183,338-444,678-691
//
// Design (see DESIGN.md §4.1):
//   * activations NHWC bf16; one tile = 16 rows x 8 cols of output positions (M = 128);
//   * the A operand of every filter tap is a *row-shifted window* of a "strip" —
//     (16 + taps-1) rows x 8 cols x 64 channels — that TMA drops into shared memory once,
//     so vertical taps re-use the same bytes (rows are 1024 B = one SWIZZLE_128B atom, so
//     every window start stays atom-aligned);
//   * stride-2 convs read the input through a 5-D "phase split" view
//     (2C, W/2, 2, H/2, N) of the same NHWC buffer, stride-2 transposed convs write their
//     output through the same view — no im2col, no scatter kernels;
//   * a work item is a PAIR of tiles of the same (variant, n-tile) when the accumulator is
//     <= 128 columns wide: every weight k-block that TMA brings in feeds two M=128 MMAs
//     (M = 256 per CTA per B stage), and the TMEM holds two such pairs (4 x 128 columns) so the
//     epilogue of one item overlaps the MMAs of the next; wider accumulators (<= 256
//     columns) run as single tiles, double-buffered the same way;
//   * a per-layer *program* (strips -> taps) built on the host drives three warp-uniform roles
//     (A producer, B producer, MMA issuer); 16 epilogue warps (four groups splitting the
//     channels) drain the accumulators: +bias, activation, optional GDN — the squared tile goes
//     to smem as a bf16 A operand, a second tcgen05.mma against gamma' writes the norm IN PLACE
//     over the accumulator while x stays in registers — optional per-pixel scale, then
//     swizzled smem staging and a TMA store.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/masic_b200.h"
#include "cvt16.cuh"
#include "ptx.cuh"

namespace masic {

constexpr int TILE_W = 8;
constexpr int TILE_H = 16;
constexpr int KBLK = 64;            // channels per k-block: 128 B of bf16 = one swizzle row
constexpr int NUM_THREADS = 640;    // warp 0: A producer, 1: B producer, 2: MMA issuer of slot 0, 3: TMEM alloc + issuer of slot 1;
                                    // warps 4-19: four epilogue groups of 4 warps
                                    // (warp % 4 = the TMEM lane quarter a warp may read)
constexpr int EPI_THREADS = 512;
constexpr int MAX_VARIANTS = 4;
constexpr int MAX_STAGES = 8;
constexpr int MAX_STRIPS = 64, MAX_BOPS = 128;
constexpr int STAGE_BLK_BYTES = 16384;  // one 128-row x 128-B staging block
constexpr uint32_t TMEM_COLS = 512;

// One A strip of the per-tile program and the taps (MMA groups) that read it.
struct Strip {
  int16_t c0, dx, p2, dy;   // TMA coordinates relative to the tile origin
  uint8_t n_taps;           // MMA groups fed by this strip (one B k-block each)
  int8_t a_row0, a_step;    // strip row of tap j = a_row0 + j * a_step
  uint8_t nk;               // low nibble: K=16 steps per tap, high nibble: first step
};

struct Variant {
  int strip_off, n_strips, bop_off, n_bops;
  int out_p2;   // phase-row coordinate in the 5-D output view
  int out_c0;   // channel offset inside the output view (px * Cpitch)
};

struct KParams {
  CUtensorMap tmA, tmB, tmO, tmG;
  // per-layer programs live in the kernel-parameter constant bank: the role loops read them with
  // warp-uniform indices
  Strip strips[MAX_STRIPS];
  int32_t bops[MAX_BOPS];          // first row of the tap's k-block in the packed weights
  Variant var[MAX_VARIANTS];
  int n_var;
  int tiles_x, tiles_y, n_img, n_ntiles;
  int n_spatial;                   // tiles_x * tiles_y * n_img
  int n_tiles_total;               // n_spatial * n_var * n_ntiles; tile id u = group * n_spatial + s
  int n_tile;
  int pair;                        // accumulator slots per CTA and work item: 2 (n_tile <= 128) or 1
  int pdl;                         // 1: launched with programmatic stream serialization
  int b_resident;                  // 1: every weight k-block of the (single) program stays in smem for the whole kernel
  int cg2;                         // 1: launched as CTA pairs (clusters of 2) issuing tcgen05.mma.cta_group::2
  int strip_bytes, b_stage_bytes, a_stages, b_stages;
  int smem_b_off, smem_g_off, smem_stage_off, smem_misc_off;
  const float* bias;
  const float* beta;
  int gdn, out_fp32;
  int blk_ch;      // channels per staging block / TMA store
  int blk_pitch;   // bytes per row of a staging block (128 = swizzled)
  float slope[32]; // per n-tile activation: out = max(x,0) + slope * min(x,0)
  int out_coff;
  const float* rowscale;
  int rs_stride, rs_off, rs_H, rs_W;
  const __nv_bfloat16* res0;       // optional residuals added after the activation (ResidualBlock / Enhancement_Block):
  const __nv_bfloat16* res1;       // NHWC bf16, same spatial size as the output
  int res0_pitch, res0_coff, res1_pitch, res1_coff;
  int nt_in_coff[32];              // grouped launches: per n-tile input-channel offset,
  int nt_out_c[32];                // output channel position (default nt * n_tile)
  int nt_out_img[32];              // and output image offset
  int blk_img;                     // 1: staging block j of a tile goes to output image tn * nblk + j (planar / NCHW output)
  uint32_t idesc;
  uint32_t idesc_norm;   // the GDN norm MMA always runs on bf16 operands (x^2 rounded on the ALU pipe, gamma' bf16)
  int f16;         // 16-bit operand / activation format: 0 = bf16, 1 = fp16 (cvt16.cuh)
  int gdn2;        // 1: EPI_GDN2 (two epilogue teams, resident weights, one tile per item)
  __nv_bfloat16* act_out;          // EPI_RESA: act(conv + bias) before the residual adds (masic_conv_plan_set_act_out)
  int ao_pitch, ao_coff;
};

// misc smem region layout (byte offsets from smem_misc_off)
constexpr int MISC_A_FULL = 0;                       // [8] x u64
constexpr int MISC_A_EMPTY = 64;
constexpr int MISC_B_FULL = 128;
constexpr int MISC_B_EMPTY = 192;
constexpr int MISC_ACC_FULL = 256;                   // 2 x u64
constexpr int MISC_ACC_EMPTY = 272;                  // 2 x u64
constexpr int MISC_GDN_BAR = 288;
constexpr int MISC_G_FULL = 296;
constexpr int MISC_TMEM_PTR = 304;
constexpr int MISC_A2_READY = 312;                   // CTA pairs: both CTAs have written their A2 operand
constexpr int MISC_BIAS = 512;                       // 128 floats (GDN layers: bias of the single n-tile)
constexpr int MISC_BETA = 1024;                      // 128 floats
constexpr int MISC_BYTES = 1536;

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c),
               "r"(d)
               : "memory");
}
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// packed fp32 pairs (FADD2 / FMUL2 / FFMA2 on sm_100a): the epilogue is instruction-issue bound, so every
// bias add / square / scale works on two channels per instruction
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t pk2u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void upk2u(uint64_t v, uint32_t& lo, uint32_t& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint32_t pack16x2_p(uint64_t v, int f16) {   // 16-bit pair {lo, hi} of a packed fp32 pair
  float lo, hi;
  upk2(v, lo, hi);
  return pack16x2(lo, hi, f16);
}
// Operand of the GDN norm MMA: bf16(x^2) of two non-negative fp32 values WITHOUT the XU pipe — round half up in the
// integer domain and byte-permute the two upper halves together (3 ALU instructions; an F2FP pack costs ~15 cycles of
// the XU pipe per warp, the pipe the GDN epilogues are bound by).  The norm beta' + gamma' x^2 tolerates bf16 operands:
// they contribute 3e-5 of the 1e-4 rms deviation of the fp16 engine's latents (tools/noise_analysis.py).
__device__ __forceinline__ uint32_t pack_bf16x2_alu(uint64_t v) {
  uint32_t lo, hi, r;
  upk2u(v, lo, hi);
  lo += 0x8000u;
  hi += 0x8000u;
  asm("prmt.b32 %0, %1, %2, 0x7632;" : "=r"(r) : "r"(lo), "r"(hi));
  return r;
}
template <bool F16>
__device__ __forceinline__ uint32_t pack_norm_operand(uint64_t sq) {     // the A2 operand is bf16 in both formats
  if (F16) return pack_bf16x2_alu(sq);
  return pack16x2_p(sq, 0);
}
__device__ __forceinline__ float rsqrt_approx(float x) {           // one MUFU.RSQ (rsqrtf() adds a denormal fix-up path)
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void ld_shared_p2(uint32_t addr, uint64_t& a, uint64_t& b) {   // four floats as two pairs
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}

// A work item: `cnt` consecutive tiles of the same group (variant, n-tile): up to `pair` per CTA, i.e. up to
// 2*pair for a CTA pair, where tile k of the item lives in CTA (k & 1), accumulator slot (k >> 1).
struct Item {
  int cnt;        // tiles in the item (whole CTA pair)
  int nslots;     // accumulator slots in use per CTA
  int var, nt;
  bool valid[2];  // does this CTA own a tile in slot t
  int n[2], y0[2], x0[2];
};
// Position in the tile sequence u = (variant, n-tile, image, tile row, tile column): every role walks its CTA's range
// with one division at the start and increments afterwards (the walk used to cost ~10 % of all issued instructions).
struct Cursor { int u, s, nt, var, tx, ty, n; };
__device__ __forceinline__ Cursor cursor_init(const KParams& p, int u) {
  Cursor c;
  c.u = u;
  const int g = u / p.n_spatial;
  c.s = u - g * p.n_spatial;
  c.nt = g % p.n_ntiles;
  c.var = g / p.n_ntiles;
  c.tx = c.s % p.tiles_x;
  const int r = c.s / p.tiles_x;
  c.ty = r % p.tiles_y;
  c.n = r / p.tiles_y;
  return c;
}
template <bool CG2>
__device__ __forceinline__ Item next_item(const KParams& p, Cursor& c, int u_end, int rank) {
  Item it;
  it.nt = c.nt;
  it.var = c.var;
  const int cap = CG2 ? 2 * p.pair : p.pair;
  it.cnt = min(cap, min(u_end - c.u, p.n_spatial - c.s));
  it.nslots = CG2 ? (it.cnt + 1) >> 1 : it.cnt;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    it.valid[t] = false; it.n[t] = c.n; it.y0[t] = c.ty * TILE_H; it.x0[t] = c.tx * TILE_W;
  }
#pragma unroll
  for (int k = 0; k < (CG2 ? 4 : 2); ++k) {
    if (k < it.cnt) {
      const int t = CG2 ? (k >> 1) : k;
      if (!CG2 || (k & 1) == rank) {
        it.valid[t] = true; it.n[t] = c.n; it.y0[t] = c.ty * TILE_H; it.x0[t] = c.tx * TILE_W;
      }
      if (++c.tx == p.tiles_x) { c.tx = 0; if (++c.ty == p.tiles_y) { c.ty = 0; ++c.n; } }
    }
  }
  c.u += it.cnt;
  c.s += it.cnt;
  if (c.s == p.n_spatial) {
    c.s = 0; c.tx = 0; c.ty = 0; c.n = 0;
    if (++c.nt == p.n_ntiles) { c.nt = 0; ++c.var; }
  }
  return it;
}

// EPI selects the epilogue at compile time so that each variant gets its own register allocation (the GDN epilogue
// is issue- and latency-bound: a spill there costs ~40 % on the 608x1088 layers)
constexpr int EPI_PLAIN = 0, EPI_GDN = 1, EPI_RES = 2, EPI_GDN2 = 3;
// EPI_RESA: EPI_RES that also stores the activated value before the residual adds (the training step's LeakyReLU
// backward needs its sign; act + residual rounded to bf16 does not keep it where |act| << |residual|).  bf16, no CTA pairs.
constexpr int EPI_RESA = 4;
// EPI_GDN2 (layers whose whole weight set stays in shared memory, i.e. g_a_conv1): one tile per work item, TWO epilogue
// teams of 8 warps that alternate over the items, each with its own accumulator, its own norm accumulator (the norm
// MMA no longer overwrites x, so nothing has to stay in registers across it) and its own A2 / staging blocks.  The
// per-tile chain TMEM load -> x^2 -> barrier -> norm MMA -> wait -> TMEM load -> rsqrt -> staging -> TMA store is
// latency-bound (2.7 us per tile with all 16 warps in lock step); two tiles in flight hide half of it.

template <bool CG2, int EPI, bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_tc_kernel(const __grid_constant__ KParams p) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B atoms must be 1024-B aligned in the shared window
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + p.smem_b_off;
  const uint32_t sG = smem_base + p.smem_g_off;
  const uint32_t sStage = smem_base + p.smem_stage_off;
  const uint32_t sMisc = smem_base + p.smem_misc_off;
  volatile uint32_t* tmem_ptr_s =
      reinterpret_cast<volatile uint32_t*>(smem_gen + p.smem_misc_off + MISC_TMEM_PTR);

  // warp index through a shuffle: provably warp-uniform, so ptxas keeps the role loops (which only
  // depend on blockIdx and kernel parameters) on the uniform datapath
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  // the 16-bit format is a template parameter: a run-time select costs a second (predicated-off, but issued) F2FP per
  // conversion, and F2FP shares the XU pipe with MUFU at ~15 cycles per warp instruction — the pipe that bounds the
  // GDN epilogues (ncu: xu 85 % busy on g_a_conv1)
  constexpr int f16 = F16 ? 1 : 0;
  // this CTA's (CTA pair's) contiguous, balanced range of tiles
  const int rank = CG2 ? static_cast<int>(cluster_ctarank()) : 0;
  const int unit = CG2 ? blockIdx.x >> 1 : blockIdx.x, n_units = CG2 ? gridDim.x >> 1 : gridDim.x;
  const int u_begin = static_cast<int>(static_cast<long long>(unit) * p.n_tiles_total / n_units);
  const int u_end = static_cast<int>(static_cast<long long>(unit + 1) * p.n_tiles_total / n_units);
  // mbarriers the producers credit / the epilogue releases live in the leader CTA (rank 0) of a pair
  auto leader_bar = [&](uint32_t local) -> uint32_t { return CG2 ? mapa_shared(local, 0) : local; };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmO);
    for (int i = 0; i < MAX_STAGES; ++i) {
      mbar_init(sMisc + MISC_A_FULL + 8 * i, 1);
      mbar_init(sMisc + MISC_A_EMPTY + 8 * i, p.pair);     // one commit per MMA-issuing warp
      mbar_init(sMisc + MISC_B_FULL + 8 * i, 1);
      mbar_init(sMisc + MISC_B_EMPTY + 8 * i, p.pair);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(sMisc + MISC_ACC_FULL + 8 * i, p.pair);
      mbar_init(sMisc + MISC_ACC_EMPTY + 8 * i, EPI == EPI_GDN2 ? 256 : (CG2 ? 2 * EPI_THREADS : EPI_THREADS));
    }
    mbar_init(sMisc + MISC_GDN_BAR, 1);
    mbar_init(sMisc + MISC_G_FULL, 1);
    mbar_init(sMisc + MISC_A2_READY, EPI == EPI_GDN2 ? 1 : 2);   // GDN2: the second team's norm-MMA barrier
    fence_mbar_init();
  }
  if (warp == 3) {
    if (CG2) { tmem_alloc_cg2(sMisc + MISC_TMEM_PTR, TMEM_COLS); tmem_relinquish_cg2(); }
    else { tmem_alloc(sMisc + MISC_TMEM_PTR, TMEM_COLS); tmem_relinquish(); }
  }
  if ((EPI == EPI_GDN || EPI == EPI_GDN2) && threadIdx.x >= 128) {       // the single n-tile's bias / beta' stay in smem for the whole kernel
    float* bs = reinterpret_cast<float*>(smem_gen + p.smem_misc_off + MISC_BIAS);
    float* be = reinterpret_cast<float*>(smem_gen + p.smem_misc_off + MISC_BETA);
    const int i = threadIdx.x - 128;
    if (i < 128) bs[i] = p.bias[i];
    else if (i < 256) be[i - 128] = p.beta[i - 128];
  }
  tc_fence_before();
  if (CG2) cluster_sync_all(); else __syncthreads();     // barrier inits visible to the peer before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) may
  // overlap the tail of the previous kernel in the stream; from here on we read its output.  The trigger lets
  // the NEXT kernel's CTAs be scheduled as soon as SMs free up (they block in their own griddepcontrol.wait).
  if (p.pdl) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }

  // Role loops are WARP-UNIFORM (all 32 lanes walk them, barrier waits included) and only the
  // issue instructions sit under elect_one(): tcgen05.mma / TMA are uniform-datapath instructions.
  if (warp == 0) {
    // ===================== A producer: activation strips =====================
    uint32_t st = 0, ph = 0;
    const uint32_t n_st = p.a_stages, strip_bytes = p.strip_bytes, st_bytes = p.pair * p.strip_bytes;
    for (Cursor cur = cursor_init(p, u_begin); cur.u < u_end;) {
      const Item it = next_item<CG2>(p, cur, u_end, rank);
      const int i0 = p.var[it.var].strip_off, i1 = i0 + p.var[it.var].n_strips;
      const int gc0 = p.nt_in_coff[it.nt];
      for (int i = i0; i < i1; ++i) {
        const Strip sp = p.strips[i];
        const uint32_t full = sMisc + MISC_A_FULL + 8 * st;
        mbar_wait(sMisc + MISC_A_EMPTY + 8 * st, ph ^ 1);
        if (elect_one()) {
          // the leader's barrier collects the strips of every tile of the item, whichever CTA stages them
          if (rank == 0) mbar_expect_tx(full, it.cnt * strip_bytes);
          const uint32_t fl = leader_bar(full);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            if (it.valid[t]) {
              if (CG2)
                tma_load_5d_cg2(sA + st * st_bytes + t * strip_bytes, &p.tmA, fl, sp.c0 + gc0, it.x0[t] + sp.dx, sp.p2,
                                it.y0[t] + sp.dy, it.n[t]);
              else
                tma_load_5d(sA + st * st_bytes + t * strip_bytes, &p.tmA, fl, sp.c0 + gc0, it.x0[t] + sp.dx, sp.p2,
                            it.y0[t] + sp.dy, it.n[t]);
            }
          }
        }
        __syncwarp();
        if (++st == n_st) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== B producer: weight k-blocks (+ gamma once) =====================
    if ((EPI == EPI_GDN || EPI == EPI_GDN2) && elect_one()) {
      tma_prefetch_desc(&p.tmG);
      if (CG2) {          // each CTA holds the 64 N-rows of gamma' it feeds to the pair's norm MMA
        if (rank == 0) mbar_expect_tx(sMisc + MISC_G_FULL, 2 * STAGE_BLK_BYTES);
        const uint32_t gf = leader_bar(sMisc + MISC_G_FULL);
        tma_load_2d_cg2(sG, &p.tmG, gf, 0, 64 * rank);
        tma_load_2d_cg2(sG + STAGE_BLK_BYTES / 2, &p.tmG, gf, KBLK, 64 * rank);
      } else {
        mbar_expect_tx(sMisc + MISC_G_FULL, 2 * STAGE_BLK_BYTES);
        tma_load_2d(sG, &p.tmG, sMisc + MISC_G_FULL, 0, 0);
        tma_load_2d(sG + STAGE_BLK_BYTES, &p.tmG, sMisc + MISC_G_FULL, KBLK, 0);
      }
    }
    __syncwarp();
    uint32_t st = 0, ph = 0;
    const uint32_t n_st = p.b_stages, st_bytes = p.b_stage_bytes;
    if (p.b_resident) {
      // small layers (sub-pixel deconv4, the CQE's 32/64-channel 3x3 convs): all k-blocks are loaded once, stage i
      // holds tap i for the whole kernel, and the issuers skip the per-tap full/empty handshake (with N <= 64 a tap's
      // MMAs take less time than one trip round the ring)
      if (u_begin < u_end && elect_one()) {
        const Variant& v0 = p.var[0];
        mbar_expect_tx(sMisc + MISC_B_FULL, v0.n_bops * st_bytes);
        for (int i = 0; i < v0.n_bops; ++i)
          tma_load_2d(sB + i * st_bytes, &p.tmB, sMisc + MISC_B_FULL, 0, p.bops[v0.bop_off + i]);
      }
      __syncwarp();
    } else
    for (Cursor cur = cursor_init(p, u_begin); cur.u < u_end;) {
      const Item it = next_item<CG2>(p, cur, u_end, rank);
      // a CTA of a pair stages its half of the n-tile's rows (st_bytes = that half)
      const int nrow = it.nt * p.n_tile + (CG2 ? rank * (p.n_tile >> 1) : 0);
      const int i0 = p.var[it.var].bop_off, i1 = i0 + p.var[it.var].n_bops;
      for (int i = i0; i < i1; ++i) {
        const int row0 = p.bops[i];
        const uint32_t full = sMisc + MISC_B_FULL + 8 * st;
        mbar_wait(sMisc + MISC_B_EMPTY + 8 * st, ph ^ 1);
        if (elect_one()) {
          if (rank == 0) mbar_expect_tx(full, CG2 ? 2 * st_bytes : st_bytes);
          if (CG2) tma_load_2d_cg2(sB + st * st_bytes, &p.tmB, leader_bar(full), 0, row0 + nrow);
          else tma_load_2d(sB + st * st_bytes, &p.tmB, full, 0, row0 + nrow);
        }
        __syncwarp();
        if (++st == n_st) { st = 0; ph ^= 1; }
      }
    }
  } else if ((warp == 2 || (warp == 3 && p.pair == 2)) && rank == 0) {
    // ===================== MMA issuers (CTA pairs: the leader issues for both CTAs) =====================
    // One issuing warp per accumulator slot: with two tiles per item, warp 2 feeds slot 0 and warp 3 slot 1 from
    // the SAME A/B stages, so each warp's loop (mbarrier waits, descriptor arithmetic, 4 MMAs, commits) only
    // has to keep up with half of the tensor-pipe work.  Every stage is released by one commit per issuer.
    const int slot = warp - 2;
    const uint32_t n_sa = p.a_stages, n_sb = p.b_stages;
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
    // descriptor = constant high part | (smem address >> 4); +2 per K=16 step, +64 per strip row
    const uint64_t descA0 = umma_desc_sw128(sA) + slot * (p.strip_bytes >> 4), descB0 = umma_desc_sw128(sB);
    const uint32_t a_step = (p.pair * p.strip_bytes) >> 4, b_step = p.b_stage_bytes >> 4;
    const uint32_t idesc = p.idesc;
    // with the range test folded in, b_res is a computed value that ptxas keeps in a uniform predicate; the bare
    // kernel parameter was re-read from the constant bank twice per tap of the loop below
    const bool b_res = p.b_resident != 0 && u_begin < u_end;
    if (b_res) mbar_wait(sMisc + MISC_B_FULL, 0);     // the whole weight set has landed
    int n_item = 0;
    for (Cursor cur = cursor_init(p, u_begin); cur.u < u_end; ++n_item) {
      const Item it = next_item<CG2>(p, cur, u_end, rank);
      const int buf = n_item & 1;
      mbar_wait(sMisc + MISC_ACC_EMPTY + 8 * buf, ((n_item >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d0 = tmem_base + (EPI == EPI_GDN2 ? buf * 128 : buf * 256 + slot * 128);
      const bool active = slot < it.nslots;                // an item may fill only slot 0
      uint32_t acc = 0;                                    // 0 for the first MMA group of the item
      const int i0 = p.var[it.var].strip_off, i1 = i0 + p.var[it.var].n_strips;
      for (int i = i0; i < i1; ++i) {
        const Strip sp = p.strips[i];
        const uint32_t nk = sp.nk & 15u, k0 = sp.nk >> 4;
        mbar_wait(sMisc + MISC_A_FULL + 8 * sa, pa);
        uint64_t adesc = descA0 + (sa * a_step + static_cast<uint32_t>(sp.a_row0) * 64u + 2u * k0);
        const int64_t a_inc = static_cast<int64_t>(sp.a_step) * 64;
        const int n_taps = sp.n_taps;
        for (int j = 0; j < n_taps; ++j) {
          if (!b_res) mbar_wait(sMisc + MISC_B_FULL + 8 * sb, pb);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t bdesc = descB0 + (sb * b_step + 2u * k0);
            auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t ac) {
              if (CG2) umma_bf16_cg2(d, a, b, idesc, ac); else umma_bf16(d, a, b, idesc, ac);
            };
            auto commit = [&](uint32_t bar) { if (CG2) umma_commit_cg2(bar); else umma_commit(bar); };
            if (active) {
              if (nk == 4) {
                mma(d0, adesc, bdesc, acc);
                mma(d0, adesc + 2, bdesc + 2, 1u);
                mma(d0, adesc + 4, bdesc + 4, 1u);
                mma(d0, adesc + 6, bdesc + 6, 1u);
              } else {
                for (uint32_t k = 0; k < nk; ++k) mma(d0, adesc + 2 * k, bdesc + 2 * k, k ? 1u : acc);
              }
            }
            if (!b_res) commit(sMisc + MISC_B_EMPTY + 8 * sb);
            if (j + 1 == n_taps) {
              commit(sMisc + MISC_A_EMPTY + 8 * sa);
              if (i + 1 == i1) commit(sMisc + MISC_ACC_FULL + 8 * buf);
            }
          }
          __syncwarp();
          acc = 1u;
          adesc += a_inc;
          if (++sb == n_sb) { sb = 0; pb ^= 1; }
        }
        if (++sa == n_sa) { sa = 0; pa ^= 1; }
      }
    }
  } else if (EPI == EPI_GDN2 && warp >= 4) {
    // ===================== epilogue, two teams (see EPI_GDN2 above) =====================
    // TMEM columns: accumulator of team T at 128 T, its norm at 256 + 128 T.  Team T = items with (n_item & 1) == T.
    // Inside a team: warp quarter ew reads TMEM lanes 32 ew .. 32 ew + 31 (= tile rows), half hf owns channels
    // 64 hf .. 64 hf + 63 = SWIZZLE_128B block hf of the team's two A2 / staging blocks.
    const int team = (warp - 4) >> 3;
    const int hf = ((warp - 4) >> 2) & 1;
    const int ew = warp & 3;
    const int t = ew * 32 + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(ew * 32) << 16;
    const uint32_t tbar = 1 + team;                               // named barrier of the team (256 threads)
    const bool leader = (t == 0 && hf == 0);
    const uint32_t sbuf = sStage + team * 2 * STAGE_BLK_BYTES;    // blocks 2T, 2T+1
    const uint32_t bias_s = sMisc + MISC_BIAS, beta_s = sMisc + MISC_BETA;
    const uint32_t gbar = sMisc + (team ? MISC_A2_READY : MISC_GDN_BAR);
    const bool fwd = (p.gdn == MASIC_GDN_FWD);
    const uint32_t acc_addr = tmem_base + lane_sel + team * 128;
    const uint32_t nrm_addr = tmem_base + lane_sel + 256 + team * 128;
    const uint32_t arow = sbuf + hf * STAGE_BLK_BYTES + t * 128;
    uint32_t gpar = 0;
    if (hf == 0 && ew == 0) mbar_wait(sMisc + MISC_G_FULL, 0);   // gamma' resident: the warp that issues the team's norm MMAs waits
    int n_item = 0;
    for (Cursor cur = cursor_init(p, u_begin); cur.u < u_end; ++n_item) {
      const Item it = next_item<CG2>(p, cur, u_end, rank);
      if ((n_item & 1) != team) continue;
      const Variant& v = p.var[it.var];
      mbar_wait(sMisc + MISC_ACC_FULL + 8 * team, (n_item >> 1) & 1);
      tc_fence_after();
      float rs = 1.0f;
      if (p.rowscale) {
        const int y = it.y0[0] + (t >> 3), x = it.x0[0] + (t & 7);
        if (y < p.rs_H && x < p.rs_W)
          rs = __ldg(p.rowscale + (static_cast<size_t>(it.n[0] * p.rs_H + y) * p.rs_W + x) * p.rs_stride + p.rs_off);
      }
      if (leader) tma_store_wait_read<0>();                       // the team's previous output tile has left its staging blocks
      named_bar_sync(tbar, 256);
      // ---- pass 1: A2[:, 64 hf .. +63] = 16-bit((acc + bias)^2)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int cb = hf * 64 + c * 32;
        uint32_t r[32];
        tmem_ld16(acc_addr + cb, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
        tmem_ld16(acc_addr + cb + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
        tmem_ld_wait();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          uint64_t xx[4];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint64_t b0, b1;
            ld_shared_p2(bias_s + (cb + 8 * c8 + 4 * q) * 4, b0, b1);
            xx[2 * q] = add2(pk2u(r[8 * c8 + 4 * q], r[8 * c8 + 4 * q + 1]), b0);
            xx[2 * q + 1] = add2(pk2u(r[8 * c8 + 4 * q + 2], r[8 * c8 + 4 * q + 3]), b1);
          }
          st_shared_v4(arow + (((4 * c + c8) ^ (t & 7)) << 4), pack_norm_operand<F16>(mul2(xx[0], xx[0])),
                       pack_norm_operand<F16>(mul2(xx[1], xx[1])), pack_norm_operand<F16>(mul2(xx[2], xx[2])),
                       pack_norm_operand<F16>(mul2(xx[3], xx[3])));
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      named_bar_sync(tbar, 256);
      if (hf == 0 && ew == 0) {                                 // one warp of the team; one elected lane issues the 8 MMAs
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d2 = tmem_base + 256 + team * 128;
          const uint64_t dh = umma_desc_sw128(0);
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            const uint64_t a2 = dh | (((sbuf + kb * STAGE_BLK_BYTES) & 0x3FFFFu) >> 4);
            const uint64_t g2 = dh | (((sG + kb * STAGE_BLK_BYTES) & 0x3FFFFu) >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d2, a2 + 2 * k, g2 + 2 * k, p.idesc_norm, (kb | k) ? 1u : 0u);
          }
          umma_commit(gbar);
        }
        __syncwarp();
      }
      mbar_wait(gbar, gpar);
      gpar ^= 1;
      tc_fence_after();
      // ---- pass 2: out = (acc + bias) * rsqrt(beta' + norm)   (IGDN: * sqrt); the staging rows re-use the A2 rows
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int cb = hf * 64 + c * 32;
        uint32_t r[32], nn[32];
        tmem_ld16(acc_addr + cb, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
        tmem_ld16(acc_addr + cb + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
        tmem_ld16(nrm_addr + cb, *reinterpret_cast<uint32_t(*)[16]>(&nn[0]));
        tmem_ld16(nrm_addr + cb + 16, *reinterpret_cast<uint32_t(*)[16]>(&nn[16]));
        tmem_ld_wait();
        if (c == 1) {                                             // last TMEM read of this item: the MMA warp may refill the accumulator
          tc_fence_before();
          mbar_arrive(sMisc + MISC_ACC_EMPTY + 8 * team);
        }
        const uint64_t rs2 = pk2(rs, rs);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          uint64_t o[4];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint64_t b0, b1, e0, e1;
            ld_shared_p2(bias_s + (cb + 8 * c8 + 4 * q) * 4, b0, b1);
            ld_shared_p2(beta_s + (cb + 8 * c8 + 4 * q) * 4, e0, e1);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int i0 = 8 * c8 + 4 * q + 2 * e;
              const uint64_t x = add2(pk2u(r[i0], r[i0 + 1]), e ? b1 : b0);
              const uint64_t nrm = add2(pk2u(nn[i0], nn[i0 + 1]), e ? e1 : e0);
              float n0, n1;
              upk2(nrm, n0, n1);
              uint64_t f = pk2(rsqrt_approx(n0), rsqrt_approx(n1));
              if (!fwd) f = mul2(f, nrm);
              uint64_t y = mul2(x, f);
              if (p.rowscale) y = mul2(y, rs2);
              o[2 * q + e] = y;
            }
          }
          st_shared_v4(arow + (((4 * c + c8) ^ (t & 7)) << 4), pack16x2_p(o[0], f16), pack16x2_p(o[1], f16),
                       pack16x2_p(o[2], f16), pack16x2_p(o[3], f16));
        }
      }
      fence_proxy_async_smem();
      named_bar_sync(tbar, 256);
      if (leader && it.valid[0]) {
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
          tma_store_5d(&p.tmO, sbuf + kb * STAGE_BLK_BYTES, p.out_coff + v.out_c0 + it.nt * p.n_tile + 64 * kb, it.x0[0],
                       v.out_p2, it.y0[0], it.n[0]);
        tma_store_commit();
      }
    }
    if (leader) tma_store_wait_all<0>();
  } else if (warp >= 4) {
    // ===================== epilogue: TMEM -> regs -> smem -> TMA store =====================
    // Four groups of 4 warps (16 warps keep the 4 schedulers busy while tcgen05.ld / MUFU / st.shared latencies
    // overlap).  Groups 2P and 2P+1 form a pair sharing 128-B staging rows: group g writes the 16-B chunks
    // [4*(g&1), 4*(g&1)+4) of every row.  GDN: pair P owns channels [64P, 64P+64) = staging block P (the two
    // blocks are the A2 operand of the norm MMA).  Otherwise pair P owns the channel blocks j = P, P+2, ... and
    // two staging blocks, so a block's TMA store drains behind the next block.
    const int grp = (warp - 4) >> 2;
    const int half = grp & 1, pr = grp >> 1;
    const int ew = warp & 3;            // the TMEM lane quarter this warp may read
    const int t = ew * 32 + lane;       // accumulator row = tile position
    const uint32_t lane_sel = static_cast<uint32_t>(ew * 32) << 16;
    const uint32_t pbar = 1 + pr;       // named barrier of this pair (256 threads); barrier 3 = all epilogue threads
    const bool leader = (t == 0 && half == 0);   // issues this pair's TMA stores (bulk groups are per thread)
    const int nblk = p.n_tile / p.blk_ch;
    const uint32_t sbuf = sStage + pr * (EPI == EPI_GDN ? 1 : 2) * STAGE_BLK_BYTES;
    const uint32_t bias_s = sMisc + MISC_BIAS, beta_s = sMisc + MISC_BETA;
    uint32_t flip = 0, gdn_par = 0;
    const float* __restrict__ bias_g = p.bias;
    const bool fwd = (p.gdn == MASIC_GDN_FWD);
    const int sw = (p.blk_pitch == 128) ? (t & 7) : 0;
    // plain path: a block's 16-channel chunks are split between the pair's two groups (bf16 rows hold up to 4 chunks,
    // fp32 rows 2); a group handles at most two
    const int nchunk_blk = p.blk_ch / 16;
    const int cpg = (nchunk_blk + 1) >> 1;
    int n_item = 0;
    if (EPI == EPI_GDN && rank == 0 && grp == 0 && ew == 0) mbar_wait_cluster(sMisc + MISC_G_FULL, 0);
    const uint32_t acc_empty0 = leader_bar(sMisc + MISC_ACC_EMPTY);
    auto release_acc = [&](int buf) {              // this thread has finished reading the item's accumulators
      tc_fence_before();
      if (CG2) mbar_arrive_cluster(acc_empty0 + 8 * buf); else mbar_arrive(acc_empty0 + 8 * buf);
    };
    for (Cursor cur = cursor_init(p, u_begin); cur.u < u_end; ++n_item) {
      const Item it = next_item<CG2>(p, cur, u_end, rank);
      const Variant& v = p.var[it.var];
      const int buf = n_item & 1;
      const float slope = p.slope[it.nt];
      const float* __restrict__ bias_t = bias_g ? bias_g + it.nt * p.n_tile : nullptr;
      mbar_wait(sMisc + MISC_ACC_FULL + 8 * buf, (n_item >> 1) & 1);
      tc_fence_after();
      if (EPI == EPI_GDN) {
      for (int tt = 0; tt < it.nslots; ++tt) {
        const uint32_t acc_addr = tmem_base + lane_sel + buf * 256 + tt * 128;
        const bool last_tile = (tt + 1 == it.nslots);
        // selects instead of dynamically indexed arrays (those would live in local memory)
        const bool valid = tt ? it.valid[1] : it.valid[0];   // CTA pairs: an odd item leaves the peer's last slot without a tile
        const int tn = tt ? it.n[1] : it.n[0], ty0 = tt ? it.y0[1] : it.y0[0], tx0 = tt ? it.x0[1] : it.x0[0];
        float rs = 1.0f;
        if (p.rowscale && valid) {
          const int y = ty0 + (t >> 3), x = tx0 + (t & 7);
          if (y < p.rs_H && x < p.rs_W)
            rs = __ldg(p.rowscale + (static_cast<size_t>(tn * p.rs_H + y) * p.rs_W + x) * p.rs_stride + p.rs_off);
        }
        {
          // ---- pass 1: x = acc + bias stays in registers; A2[:, 32g .. 32g+32) = bf16(x^2) (SWIZZLE_128B block pr)
          const int cb = grp * 32;
          uint32_t r[32];
          tmem_ld16(acc_addr + cb, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
          tmem_ld16(acc_addr + cb + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
          if (leader) tma_store_wait_read<0>();          // staging block pr (== A2 block pr) free again
          tmem_ld_wait();
          named_bar_sync(pbar, 256);
          const uint32_t arow = sbuf + t * 128;
          uint64_t x2[16];                                // x = acc + bias, two channels per register pair
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            uint64_t b0, b1;
            ld_shared_p2(bias_s + (cb + 4 * q) * 4, b0, b1);
            x2[2 * q] = add2(pk2u(r[4 * q], r[4 * q + 1]), b0);
            x2[2 * q + 1] = add2(pk2u(r[4 * q + 2], r[4 * q + 3]), b1);
          }
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8) {
            const uint64_t* xx = &x2[4 * c8];
            st_shared_v4(arow + (((4 * half + c8) ^ (t & 7)) << 4), pack_norm_operand<F16>(mul2(xx[0], xx[0])),
                         pack_norm_operand<F16>(mul2(xx[1], xx[1])), pack_norm_operand<F16>(mul2(xx[2], xx[2])),
                         pack_norm_operand<F16>(mul2(xx[3], xx[3])));
          }
          fence_proxy_async_smem();
          tc_fence_before();
          named_bar_sync(3, EPI_THREADS);
          if (grp == 0 && ew == 0) {                      // warp-uniform; one elected lane issues the 8 MMAs
            if (CG2) {        // the pair's norm MMA reads both CTAs' A2: tell the leader this CTA's half is in place
              if (elect_one()) mbar_arrive_cluster(leader_bar(sMisc + MISC_A2_READY));
              __syncwarp();
              if (rank == 0) mbar_wait_cluster(sMisc + MISC_A2_READY, gdn_par);
            }
            tc_fence_after();
            if (rank == 0 && elect_one()) {
              // norm = x^2 * gamma'^T written IN PLACE over the accumulator (every thread holds its x in registers)
              const uint32_t d2 = tmem_base + buf * 256 + tt * 128;
              const uint64_t dh = umma_desc_sw128(0);
#pragma unroll
              for (int kb = 0; kb < 2; ++kb) {
                const uint64_t a2 = dh | (((sStage + kb * STAGE_BLK_BYTES) & 0x3FFFFu) >> 4);
                const uint64_t g2 = dh | (((sG + kb * (CG2 ? STAGE_BLK_BYTES / 2 : STAGE_BLK_BYTES)) & 0x3FFFFu) >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  if (CG2) umma_bf16_cg2(d2, a2 + 2 * k, g2 + 2 * k, p.idesc_norm, (kb | k) ? 1u : 0u);
                  else umma_bf16(d2, a2 + 2 * k, g2 + 2 * k, p.idesc_norm, (kb | k) ? 1u : 0u);
                }
              }
              if (CG2) umma_commit_cg2(sMisc + MISC_GDN_BAR); else umma_commit(sMisc + MISC_GDN_BAR);
            }
            __syncwarp();
          }
          mbar_wait(sMisc + MISC_GDN_BAR, gdn_par);
          gdn_par ^= 1;
          tc_fence_after();
          // ---- pass 2: out[:, 32g .. 32g+32) = x * rsqrt(beta + norm)  (IGDN: x * sqrt(.))
          tmem_ld16(acc_addr + cb, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
          tmem_ld16(acc_addr + cb + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
          tmem_ld_wait();
          if (last_tile) release_acc(buf);              // last TMEM read of this item's accumulators
          // IGDN: sqrt(n) = n * rsqrt(n) on the MUFU fast path (2-ulp rsqrt is far below bf16 rounding)
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            uint64_t e0, e1;
            ld_shared_p2(beta_s + (cb + 4 * q) * 4, e0, e1);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const uint64_t nrm = add2(pk2u(r[4 * q + 2 * e], r[4 * q + 2 * e + 1]), e ? e1 : e0);
              float n0, n1;
              upk2(nrm, n0, n1);
              uint64_t f = pk2(rsqrt_approx(n0), rsqrt_approx(n1));
              if (!fwd) f = mul2(f, nrm);
              x2[2 * q + e] = mul2(x2[2 * q + e], f);
            }
          }
          if (p.rowscale) {
            const uint64_t rs2 = pk2(rs, rs);
#pragma unroll
            for (int i = 0; i < 16; ++i) x2[i] = mul2(x2[i], rs2);
          }
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8) {
            const uint64_t* xx = &x2[4 * c8];
            st_shared_v4(arow + (((4 * half + c8) ^ (t & 7)) << 4), pack16x2_p(xx[0], f16), pack16x2_p(xx[1], f16),
                         pack16x2_p(xx[2], f16), pack16x2_p(xx[3], f16));
          }
          fence_proxy_async_smem();
          named_bar_sync(pbar, 256);
          if (leader && valid) {
            tma_store_5d(&p.tmO, sbuf, p.out_coff + v.out_c0 + it.nt * p.n_tile + 64 * pr, tx0, v.out_p2, ty0,
                         tn);
            tma_store_commit();
          }
        }
      }
      } else {
        // ---- plain epilogue: bias, activation, per-pixel scale, residual adds.  The item's (tile, block) units are dealt
        // round-robin to the two group pairs, so two narrow tiles (<= 64 channels) drain concurrently.
        const int n_units = it.nslots * nblk;
        if (pr >= n_units) release_acc(buf);         // nothing to do for this group pair
        int tt = 0, j = pr;
        while (j >= nblk) { j -= nblk; ++tt; }
        for (int q = pr; q < n_units; q += 2) {
          const uint32_t acc_addr = tmem_base + lane_sel + buf * 256 + tt * 128;
          const bool valid = tt ? it.valid[1] : it.valid[0];
          const int tn = tt ? it.n[1] : it.n[0], ty0 = tt ? it.y0[1] : it.y0[0], tx0 = tt ? it.x0[1] : it.x0[0];
          float rs = 1.0f;
          size_t pix = 0;                           // linear output pixel of this thread's row (residual / rowscale)
          bool pix_ok = false;
          if ((p.rowscale || EPI == EPI_RES || EPI == EPI_RESA) && valid) {
            const int y = ty0 + (t >> 3), x = tx0 + (t & 7);
            pix_ok = y < p.rs_H && x < p.rs_W;
            pix = static_cast<size_t>(tn * p.rs_H + y) * p.rs_W + x;
            if (p.rowscale && pix_ok) rs = __ldg(p.rowscale + pix * p.rs_stride + p.rs_off);
          }
          const uint32_t sb2 = sbuf + flip * STAGE_BLK_BYTES;
          flip ^= 1;
          const int c = j * p.blk_ch;                 // first channel of the block inside the n-tile
          const uint32_t row = sb2 + t * p.blk_pitch;
          const int k0 = half * cpg;                  // this group's first 16-channel chunk of the block
          const bool has0 = k0 < nchunk_blk, has1 = cpg == 2 && k0 + 1 < nchunk_blk;
          // residual rows are fetched first: their latency hides behind the TMEM load and the pair barrier
          const bool do_res = (EPI == EPI_RES || EPI == EPI_RESA) && pix_ok;
          uint4 rv[8];
          if (do_res) {
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              if (kk == 0 ? has0 : has1) {
                const int gch = it.nt * p.n_tile + c + 16 * (k0 + kk);
                const uint4* r0 = reinterpret_cast<const uint4*>(p.res0 + pix * p.res0_pitch + p.res0_coff + gch);
                rv[4 * kk] = __ldg(r0); rv[4 * kk + 1] = __ldg(r0 + 1);
                if (p.res1) {
                  const uint4* r1 = reinterpret_cast<const uint4*>(p.res1 + pix * p.res1_pitch + p.res1_coff + gch);
                  rv[4 * kk + 2] = __ldg(r1); rv[4 * kk + 3] = __ldg(r1 + 1);
                }
              }
            }
          }
          uint32_t r[32];
          if (has0) tmem_ld16(acc_addr + c + 16 * k0, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
          if (has1) tmem_ld16(acc_addr + c + 16 * k0 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
          if (leader) tma_store_wait_read<1>();        // the store issued two blocks ago has left this buffer
          tmem_ld_wait();
          if (q + 2 >= n_units) release_acc(buf);      // this thread's last TMEM read of the item
          named_bar_sync(pbar, 256);
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            if (kk == 0 ? has0 : has1) {
              const int ch = c + 16 * (k0 + kk);       // channel inside the n-tile
              uint64_t o2[8];                          // 16 channels as packed pairs
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                o2[2 * e] = pk2u(r[16 * kk + 4 * e], r[16 * kk + 4 * e + 1]);
                o2[2 * e + 1] = pk2u(r[16 * kk + 4 * e + 2], r[16 * kk + 4 * e + 3]);
              }
              if (bias_t) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias_t + ch) + e);
                  o2[2 * e] = add2(o2[2 * e], pk2(b4.x, b4.y));
                  o2[2 * e + 1] = add2(o2[2 * e + 1], pk2(b4.z, b4.w));
                }
              }
              if (slope != 1.0f) {                     // ReLU / LeakyReLU: max(x, slope * x) for slope in [0, 1)
                const uint64_t sl2 = pk2(slope, slope);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  float a0, a1, s0, s1;
                  upk2(o2[i], a0, a1);
                  upk2(mul2(o2[i], sl2), s0, s1);
                  o2[i] = pk2(fmaxf(a0, s0), fmaxf(a1, s1));
                }
              }
              if (p.rowscale) {
                const uint64_t rs2 = pk2(rs, rs);
#pragma unroll
                for (int i = 0; i < 8; ++i) o2[i] = mul2(o2[i], rs2);
              }
              if (EPI == EPI_RESA && do_res) {         // the 16 activated channels before the residual adds
                uint4* ao = reinterpret_cast<uint4*>(p.act_out + pix * p.ao_pitch + p.ao_coff + it.nt * p.n_tile + ch);
                ao[0] = make_uint4(pack16x2_p(o2[0], f16), pack16x2_p(o2[1], f16), pack16x2_p(o2[2], f16),
                                   pack16x2_p(o2[3], f16));
                ao[1] = make_uint4(pack16x2_p(o2[4], f16), pack16x2_p(o2[5], f16), pack16x2_p(o2[6], f16),
                                   pack16x2_p(o2[7], f16));
              }
              if (do_res) {                            // out += residual(s): 16 bf16 = two 16-byte words each
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                  if (rr == 1 && !p.res1) continue;
                  const uint4 u0 = rv[4 * kk + 2 * rr], u1 = rv[4 * kk + 2 * rr + 1];
                  const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
                  for (int e = 0; e < 8; ++e) {
                    const float2 f = unpack16x2(w[e], f16);
                    o2[e] = add2(o2[e], pk2(f.x, f.y));
                  }
                }
              }
              if (p.out_fp32) {
                const int ch16 = 4 * (k0 + kk);        // 16 fp32 = four 16-B chunks
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  uint32_t w0, w1, w2, w3;
                  upk2u(o2[2 * e], w0, w1);
                  upk2u(o2[2 * e + 1], w2, w3);
                  st_shared_v4(row + (((ch16 + e) ^ sw) << 4), w0, w1, w2, w3);
                }
              } else {
                const int ch16 = 2 * (k0 + kk);        // 16 bf16 = two 16-B chunks
#pragma unroll
                for (int e = 0; e < 2; ++e)
                  st_shared_v4(row + (((ch16 + e) ^ sw) << 4), pack16x2_p(o2[4 * e], f16), pack16x2_p(o2[4 * e + 1], f16),
                               pack16x2_p(o2[4 * e + 2], f16), pack16x2_p(o2[4 * e + 3], f16));
              }
            }
          }
          fence_proxy_async_smem();
          named_bar_sync(pbar, 256);
          if (leader && valid) {
            if (p.blk_img)
              tma_store_5d(&p.tmO, sb2, p.out_coff + v.out_c0 + p.nt_out_c[it.nt], tx0, v.out_p2, ty0, tn * nblk + j);
            else
              tma_store_5d(&p.tmO, sb2, p.out_coff + v.out_c0 + p.nt_out_c[it.nt] + c, tx0, v.out_p2, ty0,
                           tn + p.nt_out_img[it.nt]);
            tma_store_commit();
          }
          j += 2;                                      // next unit of this pair: (tt, j) advances by two blocks
          while (j >= nblk) { j -= nblk; ++tt; }
        }
      }
    }
    if (leader) tma_store_wait_all<0>();
  }

  tc_fence_before();
  if (CG2) cluster_sync_all(); else __syncthreads();     // no CTA leaves while its peer may still signal it
  if (warp == 3) {
    tc_fence_after();
    if (CG2) tmem_dealloc_cg2(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ===================================================================== host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 5-D view (sx*Cp, W/sx, sy, H/sy, N) of an NHWC buffer; sx = sy = 1 gives (Cp, W, 1, H, N).
static int encode_nhwc_view(CUtensorMap* tm, const void* base, int elem_bytes, int n, int h, int w,
                            int cp, int split, int box_c, int box_rows, bool swizzle) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MASIC_EDRIVER;
  const int s = split ? 2 : 1;
  if (h % s || w % s) return MASIC_EINVAL;
  cuuint64_t dims[5] = {(cuuint64_t)s * cp, (cuuint64_t)(w / s), (cuuint64_t)s, (cuuint64_t)(h / s),
                        (cuuint64_t)n};
  const cuuint64_t e = elem_bytes;
  cuuint64_t strides[4] = {(cuuint64_t)s * cp * e, (cuuint64_t)w * cp * e,
                           (cuuint64_t)s * w * cp * e, (cuuint64_t)h * w * cp * e};
  cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)TILE_W, 1, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  for (int i = 0; i < 4; ++i)
    if (strides[i] % 16) return MASIC_EINVAL;
  if (reinterpret_cast<uintptr_t>(base) % 16) return MASIC_EINVAL;
  CUresult r = enc(tm, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                   5, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MASIC_OK : MASIC_EDRIVER;
}

static int encode_rows64(CUtensorMap* tm, const void* base, long rows, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MASIC_EDRIVER;
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MASIC_OK : MASIC_EDRIVER;
}
// MASIC_CONV_XFOLD4 input: a [N][H][W + MASIC_IMG_XPAD][16] bf16 image (pixel x at column x + MASIC_IMG_XOFF, pad
// columns zero) seen as OVERLAPPING 4-pixel windows: dims (64 elements, (W+XPAD)/2 windows 64 B apart, 2 row phases,
// H/2, N).  Window hx starts at column 2*hx, i.e. pixel 2*hx - 2.
static int encode_xfold4_view(CUtensorMap* tm, const void* base, int n, int h, int w, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MASIC_EDRIVER;
  const cuuint64_t row_bytes = (cuuint64_t)(w + MASIC_IMG_XPAD) * 32;
  cuuint64_t dims[5] = {64, (cuuint64_t)(w + MASIC_IMG_XPAD) / 2 - 1, 2, (cuuint64_t)h / 2, (cuuint64_t)n};
  cuuint64_t strides[4] = {64, row_bytes, 2 * row_bytes, (cuuint64_t)h * row_bytes};
  cuuint32_t box[5] = {64, (cuuint32_t)TILE_W, 1, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if (reinterpret_cast<uintptr_t>(base) % 16 || (w % 2) || (h % 2)) return MASIC_EINVAL;
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MASIC_OK : MASIC_EDRIVER;
}

// MASIC_CONV_XFOLD8 input: a [N][H][W + MASIC_IMG_XPAD][8] bf16 image seen as OVERLAPPING 8-pixel windows: dims
// (64 elements, (W+XPAD)/2 - 3 windows 32 B apart, 2 row phases, H/2, N).  Window hx starts at column 2*hx = pixel 2*hx - 2.
static int encode_xfold8_view(CUtensorMap* tm, const void* base, int n, int h, int w, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MASIC_EDRIVER;
  const cuuint64_t row_bytes = (cuuint64_t)(w + MASIC_IMG_XPAD) * 16;
  cuuint64_t dims[5] = {64, (cuuint64_t)(w + MASIC_IMG_XPAD) / 2 - 3, 2, (cuuint64_t)h / 2, (cuuint64_t)n};
  cuuint64_t strides[4] = {32, row_bytes, 2 * row_bytes, (cuuint64_t)h * row_bytes};
  cuuint32_t box[5] = {64, (cuuint32_t)TILE_W, 1, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if (reinterpret_cast<uintptr_t>(base) % 16 || (w % 2) || (h % 2)) return MASIC_EINVAL;
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MASIC_OK : MASIC_EDRIVER;
}

// gamma [128][128] bf16 row-major, loaded as two (64 x 128-row) K-blocks
static int encode_gamma(CUtensorMap* tm, const void* base, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MASIC_EDRIVER;
  cuuint64_t dims[2] = {128, 128};
  cuuint64_t strides[1] = {256};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MASIC_OK : MASIC_EDRIVER;
}

}  // namespace masic

using namespace masic;

struct MasicConvPlan {
  KParams kp;
  void* d_tables = nullptr;
  int smem_bytes = 0;
  int grid = 0;
  int total_work = 0;
  double flops = 0, hbm_bytes = 0;
};

namespace {

struct TapList {   // live taps of one strip: (a_row, kb_tap_index)
  std::vector<std::pair<int, int>> taps;
};
struct StripSpec { int c0, dx, p2, dy; TapList tl; int nk; };   // nk: packed (first step << 4 | steps), 0 = per k-block default

inline int floordiv2(int t) { return t >= 0 ? t / 2 : -((-t + 1) / 2); }

// Build the per-variant programs.  Returns the strip height (rows) via *rows_out.
int build_programs(const MasicConvDesc& d, std::vector<Strip>& strips_out, std::vector<int32_t>& bops,
                   Variant* var, int* n_var, int* rows_out) {
  const int k = d.ksize, ncb = (d.c_in + KBLK - 1) / KBLK;
  const uint32_t mask = d.tap_mask ? d.tap_mask : 0xFFFFFFFFu;
  const int nk_last = (d.c_in - (ncb - 1) * KBLK) / 16;
  int rows = TILE_H;
  *n_var = 0;

  // one variant = for every 64-channel block, every strip with its taps (a_row must be an arithmetic sequence)
  auto emit_variant = [&](const std::vector<StripSpec>& specs, int n_cblocks, int out_p2, int out_c0) -> int {
    if (*n_var >= MAX_VARIANTS) return MASIC_ENOSUP;
    Variant& v = var[*n_var];
    v.strip_off = (int)strips_out.size();
    v.bop_off = (int)bops.size();
    v.out_p2 = out_p2;
    v.out_c0 = out_c0;
    for (int cb = 0; cb < n_cblocks; ++cb) {
      const int nk_def = (cb == n_cblocks - 1) ? nk_last : 4;
      for (const auto& st : specs) {
        const auto& taps = st.tl.taps;
        if (taps.empty()) continue;
        Strip s;
        s.c0 = (int16_t)(st.c0 + cb * KBLK); s.dx = (int16_t)st.dx; s.p2 = (int16_t)st.p2; s.dy = (int16_t)st.dy;
        s.n_taps = (uint8_t)taps.size();
        s.a_row0 = (int8_t)taps[0].first;
        s.a_step = (int8_t)(taps.size() > 1 ? taps[1].first - taps[0].first : 0);
        for (size_t i = 0; i < taps.size(); ++i) {
          if (taps[i].first != s.a_row0 + (int)i * s.a_step) return MASIC_ENOSUP;
          bops.push_back((taps[i].second * n_cblocks + cb) * d.c_out_pad);
        }
        s.nk = (uint8_t)(st.nk ? st.nk : nk_def);
        strips_out.push_back(s);
      }
    }
    v.n_strips = (int)strips_out.size() - v.strip_off;
    v.n_bops = (int)bops.size() - v.bop_off;
    if (v.n_bops == 0) return MASIC_EINVAL;
    ++*n_var;
    return MASIC_OK;
  };

  if (d.kind == MASIC_CONV || d.kind == MASIC_DECONV_S2_SUBPIX) {
    const int kk = (d.kind == MASIC_DECONV_S2_SUBPIX) ? 3 : k;
    const int stride = (d.kind == MASIC_DECONV_S2_SUBPIX) ? 1 : d.stride;
    const int pad = kk / 2;
    std::vector<StripSpec> specs;
    if (stride == 1) {
      rows = TILE_H + kk - 1;
      for (int kx = 0; kx < kk; ++kx) {
        StripSpec s{d.in_coff, kx - pad, 0, -pad, {}, 0};
        for (int ky = 0; ky < kk; ++ky)
          if (mask & (1u << (ky * kk + kx))) s.tl.taps.push_back({ky, ky * kk + kx});
        specs.push_back(s);
      }
    } else if (stride == 2) {
      // input row = 2*(oy + half) + py with t = ky - pad, half = floor(t/2), py = t - 2*half
      const int half_min = floordiv2(-pad), half_max = floordiv2(kk - 1 - pad);
      rows = TILE_H + (half_max - half_min);
      for (int kx = 0; kx < kk; ++kx) {
        const int tx = kx - pad, hx = floordiv2(tx), px = tx - 2 * hx;
        for (int py = 0; py < 2; ++py) {
          StripSpec s{d.in_coff + px * d.in_cpitch, hx, py, half_min, {}, 0};
          for (int ky = 0; ky < kk; ++ky) {
            const int ty = ky - pad, hy = floordiv2(ty);
            if (ty - 2 * hy != py) continue;
            if (mask & (1u << (ky * kk + kx))) s.tl.taps.push_back({hy - half_min, ky * kk + kx});
          }
          specs.push_back(s);
        }
      }
    } else {
      return MASIC_EINVAL;
    }
    int rc = emit_variant(specs, ncb, 0, 0);
    if (rc) return rc;
  } else if (d.kind == MASIC_CONV_XFOLD4) {
    // Overlapping-window view of a padded 16-channel image (encode_xfold4_view): window hx holds pixels
    // 2*hx-2 .. 2*hx+1 as 64 consecutive bf16.  Taps kx = 0..3 are one K=64 block read at window ox;
    // tap kx = 4 is K sub-block j=2 of window ox+1 (a single K=16 MMA).
    if (k != 5 || d.c_in != 64 || d.in_cpitch != 16 || d.in_coff != 0 || d.stride != 2 || d.tap_mask) return MASIC_EINVAL;
    rows = TILE_H + 2;
    std::vector<StripSpec> specs;
    for (int grp = 0; grp < 2; ++grp)
      for (int py = 0; py < 2; ++py) {
        StripSpec s{0, grp ? 1 : 0, py, -1, {}, grp ? (1 | (2 << 4)) : 4};
        for (int ky = py; ky < 5; ky += 2) s.tl.taps.push_back({(ky >> 1), ky * 2 + grp});
        specs.push_back(s);
      }
    int rc = emit_variant(specs, 1, 0, 0);
    if (rc) return rc;
  } else if (d.kind == MASIC_CONV_XFOLD8) {
    // 8-pixel windows of an 8-channel-pitch image (encode_xfold8_view): window ox holds pixels 2*ox-2 .. 2*ox+5, i.e.
    // taps kx = 0..4 of a kernel row are K columns 0..39 of ONE block: three K=16 MMAs per (ky) and nothing else.
    if (k != 5 || d.c_in != 64 || d.in_cpitch != 8 || d.in_coff != 0 || d.stride != 2 || d.tap_mask) return MASIC_EINVAL;
    rows = TILE_H + 2;
    std::vector<StripSpec> specs;
    for (int py = 0; py < 2; ++py) {
      StripSpec s{0, 0, py, -1, {}, 3};
      for (int ky = py; ky < 5; ky += 2) s.tl.taps.push_back({(ky >> 1), ky});
      specs.push_back(s);
    }
    int rc = emit_variant(specs, 1, 0, 0);
    if (rc) return rc;
  } else if (d.kind == MASIC_DECONV_S2) {
    if (k != 5) return MASIC_ENOSUP;
    // out[2q+py] gets taps ky = py, py+2, .. from input row q + dy, dy = 1 - (ky-py)/2
    rows = TILE_H + 2;
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        std::vector<StripSpec> specs;
        for (int kx = px; kx < 5; kx += 2) {
          const int dx = 1 - (kx - px) / 2;
          StripSpec s{d.in_coff, dx, 0, -1, {}, 0};
          for (int ky = py; ky < 5; ky += 2) {
            const int dy = 1 - (ky - py) / 2;
            if (mask & (1u << (ky * 5 + kx))) s.tl.taps.push_back({dy + 1, ky * 5 + kx});
          }
          specs.push_back(s);
        }
        int rc = emit_variant(specs, ncb, py, px * d.out_cpitch);
        if (rc) return rc;
      }
  } else {
    return MASIC_EINVAL;
  }
  *rows_out = rows;
  return MASIC_OK;
}

}  // namespace

extern "C" int masic_conv_plan_create(const MasicConvDesc* dp, MasicConvPlan** plan_out) {
  if (!dp || !plan_out) return MASIC_EINVAL;
  const MasicConvDesc& d = *dp;
  *plan_out = nullptr;
  if (d.c_in <= 0 || d.c_in % 16) return MASIC_EINVAL;
  if (d.n_tile % 16 || d.n_tile < 16 || d.n_tile > 256) return MASIC_EINVAL;
  if (d.c_out_pad % d.n_tile || d.c_out > d.c_out_pad) return MASIC_EINVAL;
  if (d.c_out_pad / d.n_tile > 32) return MASIC_EINVAL;
  // CTA pairs split the N of the M = 256 MMA and every B k-block between the two CTAs (n_tile / 2 rows each); the
  // pair kernel runs only where each half is a whole number of 16-wide N steps
  if (d.cta_pairs && d.n_tile % 32) return MASIC_EINVAL;
  if (d.in_cpitch % 8 || d.in_coff % 8 || d.out_coff % 8) return MASIC_EINVAL;
  if ((d.kind == MASIC_CONV_XFOLD4 || d.kind == MASIC_CONV_XFOLD8) && d.c_in != 64) return MASIC_EINVAL;
  if (d.out_cpitch % (d.out_fp32 ? 4 : 8)) return MASIC_EINVAL;
  if (d.ksize != 1 && d.ksize != 3 && d.ksize != 5) return MASIC_EINVAL;
  if (d.gdn && (d.n_tile != 128 || d.c_out != 128 || !d.gamma_packed || !d.beta || !d.bias)) return MASIC_EINVAL;
  const bool xfold = d.kind == MASIC_CONV_XFOLD4 || d.kind == MASIC_CONV_XFOLD8;
  if ((d.kind == MASIC_CONV || xfold) && d.stride == 2 && (d.h_in % 2 || d.w_in % 2))
    return MASIC_EINVAL;

  MasicConvPlan* pl = new MasicConvPlan();
  KParams& kp = pl->kp;
  memset(&kp, 0, sizeof(kp));

  std::vector<Strip> strips; std::vector<int32_t> bops;
  int rows = 0;
  int rc = build_programs(d, strips, bops, kp.var, &kp.n_var, &rows);
  if (rc) { delete pl; return rc; }

  // geometry of the tile grid (output positions for conv, input positions for deconv)
  int gh, gw, out_h, out_w, out_split = 0;
  if (d.kind == MASIC_CONV || xfold) {
    gh = d.stride == 2 ? d.h_in / 2 : d.h_in;
    gw = d.stride == 2 ? d.w_in / 2 : d.w_in;
    out_h = gh; out_w = gw;
  } else if (d.kind == MASIC_DECONV_S2) {
    gh = d.h_in; gw = d.w_in; out_h = 2 * gh; out_w = 2 * gw; out_split = 1;
  } else {
    gh = d.h_in; gw = d.w_in; out_h = gh; out_w = gw;
  }
  kp.tiles_x = (gw + TILE_W - 1) / TILE_W;
  kp.tiles_y = (gh + TILE_H - 1) / TILE_H;
  kp.n_img = d.n;
  kp.n_tile = d.n_tile;
  kp.n_ntiles = d.c_out_pad / d.n_tile;
  // CTA pairs (tcgen05 cta_group::2): each CTA stages half of every weight k-block and the pair issues M = 256 MMAs
  kp.cg2 = d.cta_pairs != 0;
  kp.pdl = d.pdl != 0;
  kp.idesc = kp.cg2 ? umma_idesc_bf16_m256(d.n_tile) : umma_idesc_bf16(d.n_tile);
  kp.idesc_norm = kp.idesc;
  kp.f16 = d.f16 != 0;
  if (kp.f16) kp.idesc &= ~((1u << 7) | (1u << 10));        // a_format / b_format: 1 = bf16, 0 = fp16

  // staging block: 128-B swizzled rows when the n-tile is wide enough, else one narrow block
  const int esz = d.out_fp32 ? 4 : 2;
  const int full_blk_ch = 128 / esz;
  if (d.n_tile % full_blk_ch == 0) { kp.blk_ch = full_blk_ch; kp.blk_pitch = 128; }
  else if (d.n_tile * esz < 128) { kp.blk_ch = d.n_tile; kp.blk_pitch = d.n_tile * esz; }
  else if (!d.out_fp32 && d.n_tile % 32 == 0) { kp.blk_ch = 32; kp.blk_pitch = 64; }    // e.g. 96 channels: 3 narrow blocks
  else if (d.out_fp32 && d.n_tile % 16 == 0) { kp.blk_ch = 16; kp.blk_pitch = 64; }     // e.g. 48 fp32 channels: 3 narrow blocks
  else { delete pl; return MASIC_EINVAL; }

  // work items: pairs of tiles sharing every weight k-block when two accumulators fit 256 TMEM columns
  kp.pair = (d.n_tile <= 128) ? 2 : 1;
  // EPI_GDN2: fused GDN on a layer whose whole weight set (<= 6 k-blocks of 16 KB: g_a_conv1's five) stays in shared
  // memory next to gamma', four staging blocks and a double-buffered strip ring
  kp.gdn2 = d.gdn && !kp.cg2 && kp.n_var == 1 && kp.var[0].n_bops <= 6;
  if (kp.gdn2) kp.pair = 1;
  kp.n_spatial = kp.tiles_x * kp.tiles_y * kp.n_img;
  kp.n_tiles_total = kp.n_spatial * kp.n_var * kp.n_ntiles;

  // shared memory carve-up
  kp.strip_bytes = rows * 1024;
  kp.b_stage_bytes = (kp.cg2 ? d.n_tile / 2 : d.n_tile) * 128;      // per CTA
  const int a_stage_bytes = kp.pair * kp.strip_bytes;
  // staging: with GDN two blocks (together the A2 operand of the norm MMA, then the output tile);
  // otherwise two per epilogue group so a block's TMA store drains behind the next block
  const int n_stage_blk = (d.gdn && !kp.gdn2) ? 2 : 4;
  const int gamma_bytes = d.gdn ? (kp.cg2 ? STAGE_BLK_BYTES : 2 * STAGE_BLK_BYTES) : 0;
  const int fixed = gamma_bytes + n_stage_blk * STAGE_BLK_BYTES + MISC_BYTES + 1024 /*align*/;
  const int budget = 227 * 1024 - fixed;                      // ring bytes
  int sa = 2, sb = 2;
  // resident weights: single program, single n-tile, and the whole k-block list fits next to a double-buffered A ring
  const int n_bops0 = kp.var[0].n_bops;
  kp.b_resident = !kp.cg2 && kp.n_var == 1 && kp.n_ntiles == 1 && (d.n_tile <= 64 || kp.gdn2) &&
                  2 * a_stage_bytes + n_bops0 * kp.b_stage_bytes <= budget;
  if (kp.gdn2 && !kp.b_resident) { delete pl; return MASIC_EINVAL; }
  if (kp.b_resident) sb = n_bops0;
  if (sa * a_stage_bytes + sb * kp.b_stage_bytes > budget) { delete pl; return MASIC_EINVAL; }
  // deepen the rings with what is left (B first: a B stage is consumed by a single tap)
  for (bool grew = true; grew;) {
    grew = false;
    if (!kp.b_resident && sb < MAX_STAGES && sb < 6 && sa * a_stage_bytes + (sb + 1) * kp.b_stage_bytes <= budget) { ++sb; grew = true; }
    if (sa < 4 && (sa + 1) * a_stage_bytes + sb * kp.b_stage_bytes <= budget) { ++sa; grew = true; }
  }
  kp.a_stages = sa; kp.b_stages = sb;
  kp.smem_b_off = sa * a_stage_bytes;
  kp.smem_g_off = kp.smem_b_off + sb * kp.b_stage_bytes;
  kp.smem_stage_off = kp.smem_g_off + gamma_bytes;
  kp.smem_misc_off = kp.smem_stage_off + n_stage_blk * STAGE_BLK_BYTES;
  pl->smem_bytes = kp.smem_misc_off + MISC_BYTES + 1024;
  if (pl->smem_bytes < 120 * 1024) pl->smem_bytes = 120 * 1024;   // keep 1 CTA/SM: 512 TMEM cols each

  // tensor maps
  const int split_in = ((d.kind == MASIC_CONV || xfold) && d.stride == 2) ? 1 : 0;
  if (d.kind == MASIC_CONV_XFOLD4) rc = encode_xfold4_view(&kp.tmA, d.in, d.n, d.h_in, d.w_in, rows);
  else if (d.kind == MASIC_CONV_XFOLD8) rc = encode_xfold8_view(&kp.tmA, d.in, d.n, d.h_in, d.w_in, rows);
  else rc = encode_nhwc_view(&kp.tmA, d.in, 2, d.n, d.h_in, d.in_row_pixels ? d.in_row_pixels : d.w_in, d.in_cpitch,
                             split_in, KBLK, rows, true);
  const int ktaps = (d.kind == MASIC_DECONV_S2_SUBPIX) ? 9 : (d.kind == MASIC_CONV_XFOLD4 ? 10 : (d.kind == MASIC_CONV_XFOLD8 ? 5 : d.ksize * d.ksize));
  const int ncb = xfold ? 1 : (d.c_in + KBLK - 1) / KBLK;
  if (!rc) rc = encode_rows64(&kp.tmB, d.w_packed, (long)ktaps * ncb * d.c_out_pad, kp.cg2 ? d.n_tile / 2 : d.n_tile);
  const bool grouped = d.nt_in_coff || d.nt_out_coff || d.nt_out_img;
  // planar output: the n-tile's staging blocks are separate output images (channel planes of an NCHW tensor seen as
  // [n * nblk][H][W][out_cpitch]); wider rows than w_in on the input side only make sense for stride-1 convolutions
  kp.blk_img = d.out_blk_images != 0;
  if (kp.blk_img && (grouped || d.gdn || d.residual0 || kp.n_ntiles != 1 || d.kind != MASIC_CONV)) { delete pl; return MASIC_EINVAL; }
  if (d.in_row_pixels && (d.in_row_pixels < d.w_in || d.kind != MASIC_CONV || d.stride != 1)) { delete pl; return MASIC_EINVAL; }
  if (grouped && (!d.nt_in_coff || !d.nt_out_coff || !d.nt_out_img || d.out_images < d.n || d.gdn || d.residual0 ||
                  d.rowscale || xfold)) { delete pl; return MASIC_EINVAL; }
  for (int i = 0; i < kp.n_ntiles; ++i) {
    kp.nt_in_coff[i] = grouped ? d.nt_in_coff[i] : 0;
    kp.nt_out_c[i] = grouped ? d.nt_out_coff[i] : i * d.n_tile;
    kp.nt_out_img[i] = grouped ? d.nt_out_img[i] : 0;
    if (kp.nt_in_coff[i] % 8 || kp.nt_out_c[i] % (d.out_fp32 ? 4 : 8) || kp.nt_out_img[i] < 0 ||
        (grouped && kp.nt_out_img[i] + d.n > d.out_images)) { delete pl; return MASIC_EINVAL; }
  }
  if (!rc) rc = encode_nhwc_view(&kp.tmO, d.out, esz, grouped ? d.out_images : (kp.blk_img ? d.n * (d.n_tile / kp.blk_ch) : d.n),
                                 out_h, out_w, d.out_cpitch, out_split,
                                 kp.blk_ch, TILE_H, kp.blk_pitch == 128);
  if (!rc && d.gdn) rc = encode_gamma(&kp.tmG, d.gamma_packed, kp.cg2 ? 64 : 128);
  if (rc) { delete pl; return rc; }

  // the programs travel in the kernel parameters (constant bank)
  if (strips.size() > MAX_STRIPS || bops.size() > MAX_BOPS) { delete pl; return MASIC_ENOSUP; }
  memcpy(kp.strips, strips.data(), strips.size() * sizeof(Strip));
  memcpy(kp.bops, bops.data(), bops.size() * sizeof(int32_t));
  cudaError_t ce = cudaSuccess;

  kp.bias = d.bias; kp.beta = d.beta; kp.gdn = d.gdn; kp.out_fp32 = d.out_fp32;
  for (int i = 0; i < 32; ++i)
    kp.slope[i] = d.act[i] == MASIC_ACT_RELU ? 0.0f : (d.act[i] == MASIC_ACT_LEAKY ? 0.01f : 1.0f);
  kp.out_coff = d.out_coff;
  kp.rowscale = d.rowscale; kp.rs_stride = d.rs_stride; kp.rs_off = d.rs_off;
  kp.rs_H = gh; kp.rs_W = gw;
  if (d.residual0) {
    if (d.kind != MASIC_CONV || d.stride != 1 || d.gdn || d.res0_cpitch % 8 || d.res0_coff % 8 ||
        (d.residual1 && (d.res1_cpitch % 8 || d.res1_coff % 8))) { delete pl; return MASIC_EINVAL; }
    kp.res0 = static_cast<const __nv_bfloat16*>(d.residual0); kp.res0_pitch = d.res0_cpitch; kp.res0_coff = d.res0_coff;
    kp.res1 = static_cast<const __nv_bfloat16*>(d.residual1); kp.res1_pitch = d.res1_cpitch; kp.res1_coff = d.res1_coff;
  } else if (d.residual1) { delete pl; return MASIC_EINVAL; }
  pl->total_work = kp.n_tiles_total;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  pl->grid = pl->total_work < sms ? pl->total_work : sms;
  if (kp.cg2) {          // one work range per CTA pair; a pair handles at least two tiles at a time
    int pairs = (pl->total_work + 1) / 2;
    if (pairs > pl->grid / 2) pairs = pl->grid / 2;
    if (pairs < 1) pairs = 1;
    pl->grid = 2 * pairs;
  }

  // useful work: live taps only, real channels only
  {
    const uint32_t mask = d.tap_mask ? d.tap_mask : 0xFFFFFFFFu;
    int live = 0;
    for (int i = 0; i < d.ksize * d.ksize; ++i) live += (mask >> i) & 1;
    const double out_pos = (double)d.n * out_h * out_w;
    double macs;
    const double co_real = (d.kind == MASIC_DECONV_S2_SUBPIX) ? d.c_out / 4 : d.c_out;
    if (xfold) macs = out_pos * 25.0 * 3.0 * d.c_out;       // the real 3-channel 5x5
    else if (d.kind == MASIC_CONV) macs = out_pos * live * d.c_in * d.c_out;
    else macs = (double)d.n * d.h_in * d.w_in * 25.0 * d.c_in * co_real;   // each input feeds 25 taps
    pl->flops = 2.0 * macs + (d.gdn ? 2.0 * out_pos * 128.0 * 128.0 : 0.0);
    const double out_ch = (d.kind == MASIC_DECONV_S2_SUBPIX) ? d.c_out_pad : d.c_out;
    pl->hbm_bytes = (double)d.n * d.h_in * d.w_in * (d.kind == MASIC_CONV_XFOLD4 ? 16 : (d.kind == MASIC_CONV_XFOLD8 ? 8 : d.c_in)) * 2.0 + out_pos * out_ch * esz +
                    (double)ktaps * ncb * d.c_out_pad * 128.0;
  }

  static bool attr_set = false;
  if (!attr_set) {
#define MASIC_K2(C, E) (const void*)conv_tc_kernel<C, E, false>, (const void*)conv_tc_kernel<C, E, true>
    const void* fns[15] = {MASIC_K2(false, EPI_PLAIN), MASIC_K2(false, EPI_GDN), MASIC_K2(false, EPI_RES),
                           MASIC_K2(true, EPI_PLAIN),  MASIC_K2(true, EPI_GDN),  MASIC_K2(true, EPI_RES),
                           MASIC_K2(false, EPI_GDN2), (const void*)conv_tc_kernel<false, EPI_RESA, false>};
#undef MASIC_K2
    for (int i = 0; i < 15 && ce == cudaSuccess; ++i)
      ce = cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (ce != cudaSuccess) { delete pl; return (int)ce; }
    attr_set = true;
  }
  *plan_out = pl;
  return MASIC_OK;
}

extern "C" int masic_conv_plan_launch(const MasicConvPlan* pl, void* stream) {
  if (!pl) return MASIC_EINVAL;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(pl->grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = pl->smem_bytes;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (pl->kp.pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (pl->kp.cg2) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr; cfg.numAttrs = na;
  const int epi = pl->kp.gdn ? (pl->kp.gdn2 ? EPI_GDN2 : EPI_GDN) : (pl->kp.res0 ? EPI_RES : EPI_PLAIN);
  const bool f16 = pl->kp.f16 != 0;
#define MASIC_LAUNCH(C, E) \
  return f16 ? (int)cudaLaunchKernelEx(&cfg, conv_tc_kernel<C, E, true>, pl->kp) \
             : (int)cudaLaunchKernelEx(&cfg, conv_tc_kernel<C, E, false>, pl->kp)
  if (pl->kp.cg2) {
    if (epi == EPI_GDN) { MASIC_LAUNCH(true, EPI_GDN); }
    if (epi == EPI_RES) { MASIC_LAUNCH(true, EPI_RES); }
    MASIC_LAUNCH(true, EPI_PLAIN);
  }
  if (pl->kp.act_out) return (int)cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, EPI_RESA, false>, pl->kp);
  if (epi == EPI_GDN2) { MASIC_LAUNCH(false, EPI_GDN2); }
  if (epi == EPI_GDN) { MASIC_LAUNCH(false, EPI_GDN); }
  if (epi == EPI_RES) { MASIC_LAUNCH(false, EPI_RES); }
  MASIC_LAUNCH(false, EPI_PLAIN);
#undef MASIC_LAUNCH
}

extern "C" int masic_conv_plan_set_act_out(MasicConvPlan* pl, void* act_out_bf16, int cpitch, int coff) {
  if (!pl || !act_out_bf16 || cpitch % 8 || coff % 8 || coff < 0) return MASIC_EINVAL;
  const KParams& k = pl->kp;
  if (!k.res0 || k.out_fp32 || k.rowscale) return MASIC_EINVAL;
  if (k.cg2 || k.f16 || k.pdl || k.blk_img) return MASIC_ENOSUP;
  if (coff + k.n_ntiles * k.n_tile > cpitch) return MASIC_EINVAL;
  pl->kp.act_out = static_cast<__nv_bfloat16*>(act_out_bf16);
  pl->kp.ao_pitch = cpitch;
  pl->kp.ao_coff = coff;
  return MASIC_OK;
}

extern "C" void masic_conv_plan_destroy(MasicConvPlan* pl) {
  if (!pl) return;
  if (pl->d_tables) cudaFree(pl->d_tables);
  delete pl;
}

// The clock64() tracing hooks of the first kernel generation were removed from the hot loops.
extern "C" int masic_conv_plan_trace(const MasicConvPlan* pl, long long* out_host) {
  (void)pl; (void)out_host;
  return MASIC_ENOSUP;
}

extern "C" int masic_conv_plan_info(const MasicConvPlan* pl, double* flops, double* hbm_bytes,
                                    int* n_work_items, int* smem_bytes) {
  if (!pl) return MASIC_EINVAL;
  if (flops) *flops = pl->flops;
  if (hbm_bytes) *hbm_bytes = pl->hbm_bytes;
  if (n_work_items) *n_work_items = pl->total_work;
  if (smem_bytes) *smem_bytes = pl->smem_bytes;
  return MASIC_OK;
}
