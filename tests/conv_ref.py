"""Float64 reference of one tensor-core conv plan (a MasicConvDesc) and a per-element error bound for its output.

`reference(...)` takes the keyword arguments of `convplan.ConvPlan` (the operands as the kernel sees them: the 16-bit
input, residual and output buffers, fp32 torch-layout weights and bias, fp32 rowscale) and returns the whole output
buffer as the plan must leave it: computed values in the channels and images the plan writes, the buffer's previous
contents everywhere else.  Weights are rounded to the plan's 16-bit format first, as masic_pack_conv_weights does; bias
and rowscale stay fp32.  For fused GDN / IGDN it takes the effective beta' (fp32) and gamma' (bf16), as the kernel
reads them, and applies the kernel's documented rounding of the norm operand: x^2 is formed in fp32 and rounded to
bf16, to nearest even in the bf16 instantiations and half-up on the integer bits (pack_bf16x2_alu) in the fp16 ones.

`bound(r)` is the per-element tolerance  u |ref| + C_ACC S + C_GDN |ref|  (+ half the smallest fp16 subnormal):
  u      half an ulp of the output format relative to the value: 2^-8 bf16, 2^-11 fp16, 0 for fp32 output;
  S      the same chain run on |x|, |w|, |bias| and |rowscale| plus the residual magnitudes, times the GDN factor: it
         scales the error of the fp32 accumulation and of the fp32 epilogue arithmetic;
  C_GDN  rsqrt.approx, the fp32 norm accumulation, and the rare x^2 that rounds to the other side of a tie because
         its fp32 x differs from the exact one; 0 without GDN.
Every kernel output is one 16-bit rounding of an fp32 value whose only error is that accumulation, so the bound sits
about one output ulp above the exact result; a mistake in the epilogue or the tile walk moves an element by far more.
fp16 outputs are saturating (cvt.rn.satfinite), so the reference clamps them to +-65504.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

# constants of masic_b200/_lib.py, restated so the module imports without the CUDA library
ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
GDN_NONE, GDN_FWD, GDN_INV = 0, 1, 2
CONV, DECONV_S2, DECONV_S2_SUBPIX, CONV_XFOLD4, CONV_XFOLD8 = 0, 1, 2, 3, 4
IMG_XOFF, IMG_XPAD = 2, 8
F16_MAX = 65504.0
LEAKY_SLOPE = float(np.float32(0.01))      # the kernel's slope is the fp32 constant 0.01f

# Bound constants, set from a B200 run of tests/test_conv_tc_variants_gpu.py (NVIDIA B200, 1000 W power limit).
# C_ACC: the fp32-output cases, where the accumulation is the only error, reached 0.13 of C_ACC * S (every instantiation,
# both formats), i.e. the accumulation error stayed below 2^-21 S.
# C_GDN: the GDN / IGDN cases with fp16 output reached 1.15 of the bound with C_GDN = 2^-12, an error of about 2^-10.2
# |ref| beyond the output rounding.  It comes from x^2 operands that round to the neighbouring bf16 value: one such
# operand moves its term of the norm by up to 2^-7 of the term and the output by half that share of the norm, so the
# constant is 2^-9.  With it the largest ratio of a GDN case was 0.66.
C_ACC = 2.0 ** -18
C_GDN = 2.0 ** -9


@dataclass
class Ref:
    ref: torch.Tensor            # float64, shape of `out`: expected buffer contents (unwritten elements = previous)
    mag: torch.Tensor            # float64: S of the bound (0 where unwritten)
    written: torch.Tensor        # bool: elements the plan writes
    out_fmt: str                 # "bf16" | "fp16" | "fp32"
    gdn: bool
    act_ref: Optional[torch.Tensor] = None       # act_out buffer (EPI_RESA), same conventions
    act_mag: Optional[torch.Tensor] = None
    act_written: Optional[torch.Tensor] = None


def fmt_of(dtype: torch.dtype) -> str:
    return {torch.bfloat16: "bf16", torch.float16: "fp16", torch.float32: "fp32"}[dtype]


def round_to(v: torch.Tensor, fmt: str) -> torch.Tensor:
    """float64 -> the value the kernel stores: fp32 first (the epilogue's arithmetic), then the 16-bit format."""
    v32 = v.to(torch.float32)
    if fmt == "fp16":
        return v32.clamp(-F16_MAX, F16_MAX).to(torch.float16).double()
    if fmt == "bf16":
        return v32.to(torch.bfloat16).double()
    return v32.double()


def _sq_operand(y: torch.Tensor, f16: bool) -> torch.Tensor:
    """bf16(x^2) of the GDN norm MMA from the float64 x: x and x^2 in fp32, then RNE (bf16 plans) or round-half-up on the
    integer bits (fp16 plans, pack_bf16x2_alu)."""
    y32 = y.to(torch.float32)
    sq = y32 * y32
    if not f16:
        return sq.to(torch.bfloat16).double()
    bits = sq.view(torch.int32).to(torch.int64)
    bits = ((bits + 0x8000) & 0xFFFF0000) & 0xFFFFFFFF
    bits = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32)
    return bits.view(torch.float32).double()


def blk_channels(n_tile: int, out_fp32: bool) -> int:
    """Channels per staging block (masic_conv_plan_create): the unit of MasicConvDesc.out_blk_images."""
    esz = 4 if out_fp32 else 2
    full = 128 // esz
    if n_tile % full == 0:
        return full
    if n_tile * esz < 128:
        return n_tile
    if not out_fp32 and n_tile % 32 == 0:
        return 32
    if out_fp32 and n_tile % 16 == 0:
        return 16
    raise ValueError(f"n_tile {n_tile} has no staging layout")


def _nchw(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 3, 1, 2)


def _conv_core(xin: torch.Tensor, w: torch.Tensor, *, kind: int, ksize: int, stride: int, tap_mask: int,
               transposed: bool, c_out: int, w_in: int) -> torch.Tensor:
    """NHWC float64 input slice -> NHWC float64 pre-bias output of the plan's kind (c_out real channels; for
    DECONV_S2_SUBPIX the 4 * c_out phase-major channels)."""
    x = _nchw(xin)
    if kind == CONV:
        wc = w.flip(2, 3).permute(1, 0, 2, 3) if transposed else w         # correlation kernel (c_out, c_in, k, k)
        if tap_mask:
            m = torch.tensor([(tap_mask >> i) & 1 for i in range(ksize * ksize)], dtype=w.dtype, device=w.device)
            wc = wc * m.view(1, 1, ksize, ksize)
        y = F.conv2d(x, wc, stride=stride, padding=ksize // 2)
        y = y[..., :w_in if stride == 1 else w_in // 2]                       # in_row_pixels: only w_in columns
    elif kind in (DECONV_S2, DECONV_S2_SUBPIX):
        assert transposed and ksize == 5 and not tap_mask
        y = F.conv_transpose2d(x, w, stride=2, padding=2, output_padding=1)
        if kind == DECONV_S2_SUBPIX:                                          # [n][h][w][(py, px, co)]
            n, _, h2, w2 = y.shape
            y = y.view(n, c_out, h2 // 2, 2, w2 // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(n, 4 * c_out, h2 // 2, w2 // 2)
    else:                                # XFOLD4 / 8: pixel ox reads buffer columns 2 ox + kx (pixel 2 ox - 2 + kx)
        assert not transposed and ksize == 5 and stride == 2 and not tap_mask
        y = F.conv2d(x[:, :w.shape[1]], w, stride=2, padding=(2, 0))[..., :w_in // 2]
    return y.permute(0, 2, 3, 1)


def reference(*, kind: int = CONV, ksize: int, stride: int = 1, tap_mask: int = 0, x: torch.Tensor, in_coff: int = 0,
              c_in: int, weight: torch.Tensor, transposed: bool = False, bias: Optional[torch.Tensor] = None,
              c_out: int, n_tile: int, c_out_pad: Optional[int] = None, out: torch.Tensor, out_coff: int = 0,
              act=ACT_NONE, gdn: int = GDN_NONE, beta_p: Optional[torch.Tensor] = None,
              gamma_p: Optional[torch.Tensor] = None, rowscale: Optional[torch.Tensor] = None, rs_off: int = 0,
              residual0: Optional[torch.Tensor] = None, res0_coff: int = 0,
              residual1: Optional[torch.Tensor] = None, res1_coff: int = 0,
              nt_in_coff: Optional[Sequence[int]] = None, nt_out_coff: Optional[Sequence[int]] = None,
              nt_out_img: Optional[Sequence[int]] = None, w_in: Optional[int] = None, out_blk_images: bool = False,
              act_out: Optional[torch.Tensor] = None, act_out_coff: int = 0, **_ignored) -> Ref:
    """Expected contents of `out` (and `act_out`) after one launch of the plan these arguments describe.
    `x`, `out`, `residual*`, `act_out` are the plan's buffers before the launch; `weight` / `bias` are the fp32 torch
    tensors given to PackedConv (XFOLD: (c_out, c, 5, 5) over the c real channels; DECONV_S2_SUBPIX: the real c_out
    and bias); `beta_p` / `gamma_p` the effective GDN parameters (PackedConv.beta / .gamma16).  Extra keyword
    arguments of ConvPlan (cta_pairs, pdl, ...) do not change the result and are ignored."""
    f16 = x.dtype == torch.float16
    dt16 = torch.float16 if f16 else torch.bfloat16
    dd = dict(dtype=torch.float64, device=x.device)
    out_fmt = fmt_of(out.dtype)
    eff = 4 * c_out if kind == DECONV_S2_SUBPIX else c_out
    c_out_pad = c_out_pad if c_out_pad is not None else -(-eff // n_tile) * n_tile
    n_nt = c_out_pad // n_tile
    acts = [act] * n_nt if isinstance(act, int) else list(act)
    assert len(acts) == n_nt
    n, h_in, row_px, _ = x.shape
    xfold = kind in (CONV_XFOLD4, CONV_XFOLD8)
    if xfold:
        w_log = row_px - IMG_XPAD
    else:
        w_log = row_px if w_in is None else w_in

    wq = weight.detach().to(dt16).to(**dd)
    wa = wq.abs()
    xq = x.detach().to(**dd)
    grouped = nt_in_coff is not None or nt_out_coff is not None or nt_out_img is not None
    nt_in = list(nt_in_coff) if nt_in_coff is not None else [0] * n_nt
    nt_oc = list(nt_out_coff) if nt_out_coff is not None else [t * n_tile for t in range(n_nt)]
    nt_oi = list(nt_out_img) if nt_out_img is not None else [0] * n_nt

    def conv(xv, wv):
        kw = dict(kind=kind, ksize=ksize, stride=stride, tap_mask=tap_mask, transposed=transposed, c_out=c_out,
                  w_in=w_log)
        if xfold:
            return _conv_core(xv, wv, **kw)
        if not grouped:
            return _conv_core(xv[..., in_coff:in_coff + c_in], wv, **kw)
        parts = []                                     # n-tile t reads [in_coff + nt_in_coff[t], + c_in)
        wpad = torch.zeros((c_out_pad,) + tuple(wv.shape[1:]), **dd)
        wpad[:c_out] = wv
        for t in range(n_nt):
            c0 = in_coff + nt_in[t]
            parts.append(_conv_core(xv[..., c0:c0 + c_in], wpad[t * n_tile:(t + 1) * n_tile], **{**kw, "c_out": n_tile}))
        return torch.cat(parts, dim=-1)

    acc, mag = conv(xq, wq), conv(xq.abs(), wa)
    if acc.shape[-1] < c_out_pad:                      # pad channels: zero weights
        z = torch.zeros(acc.shape[:-1] + (c_out_pad - acc.shape[-1],), **dd)
        acc, mag = torch.cat([acc, z], -1), torch.cat([mag, z], -1)
    if bias is not None:
        b = torch.zeros(c_out_pad, **dd)
        bb = bias.detach().to(torch.float32).to(**dd)
        b[:eff] = bb.repeat(4) if kind == DECONV_S2_SUBPIX else bb
        acc, mag = acc + b, mag + b.abs()
    y = acc
    if gdn:
        sq = _sq_operand(y, f16)
        g = gamma_p.detach().to(torch.bfloat16).to(**dd)
        norm = sq @ g.t() + beta_p.detach().to(torch.float32).to(**dd)
        fac = norm.rsqrt() if gdn == GDN_FWD else norm.sqrt()
        y, mag = y * fac, mag * fac
    else:
        parts = []
        for t, a in enumerate(acts):
            v = y[..., t * n_tile:(t + 1) * n_tile]
            if a == ACT_RELU:
                v = v.clamp(min=0.0)
            elif a == ACT_LEAKY:
                v = torch.where(v > 0, v, v * LEAKY_SLOPE)
            parts.append(v)
        y = torch.cat(parts, -1)
    if rowscale is not None:
        rs = rowscale.detach().to(torch.float32).to(**dd)[..., rs_off:rs_off + 1]
        if kind == DECONV_S2:                          # the tile grid is the input grid: one scale per 2x2 block
            rs = rs.repeat_interleave(2, 1).repeat_interleave(2, 2)
        y, mag = y * rs, mag * rs.abs()
    act_val, act_mag = y, mag
    for r, off in ((residual0, res0_coff), (residual1, res1_coff)):
        if r is not None:
            rv = r.detach().to(**dd)[..., off:off + c_out_pad]
            y, mag = y + rv, mag + rv.abs()
    if out_fmt == "fp16":
        y = y.clamp(-F16_MAX, F16_MAX)

    def place(buf, vals, mvals, coff):
        ref = buf.detach().to(**dd).clone()
        mg = torch.zeros_like(ref)
        wr = torch.zeros(ref.shape, dtype=torch.bool, device=ref.device)
        cp = buf.shape[3]
        if out_blk_images:
            assert n_nt == 1 and not grouped
            bc = blk_channels(n_tile, buf.dtype == torch.float32)
            nblk = n_tile // bc
            keep = min(bc, cp - coff)
            v5 = ref.view(n, nblk, *ref.shape[1:])
            m5, w5 = mg.view(n, nblk, *ref.shape[1:]), wr.view(n, nblk, *ref.shape[1:])
            for j in range(nblk):
                v5[:, j, ..., coff:coff + keep] = vals[..., j * bc:j * bc + keep]
                m5[:, j, ..., coff:coff + keep] = mvals[..., j * bc:j * bc + keep]
                w5[:, j, ..., coff:coff + keep] = True
        else:
            for t in range(n_nt):
                c0 = coff + nt_oc[t]
                i0 = nt_oi[t]
                assert c0 + n_tile <= cp
                sl = (slice(i0, i0 + n), Ellipsis, slice(c0, c0 + n_tile))
                ref[sl] = vals[..., t * n_tile:(t + 1) * n_tile]
                mg[sl] = mvals[..., t * n_tile:(t + 1) * n_tile]
                wr[sl] = True
        return ref, mg, wr

    ref, mg, wr = place(out, y, mag, out_coff)
    res = Ref(ref=ref, mag=mg, written=wr, out_fmt=out_fmt, gdn=bool(gdn))
    if act_out is not None:
        res.act_ref, res.act_mag, res.act_written = place(act_out, act_val, act_mag, act_out_coff)
    return res


def bound(ref: torch.Tensor, mag: torch.Tensor, out_fmt: str, gdn: bool, c_acc: float = None,
          c_gdn: float = None) -> torch.Tensor:
    c_acc = C_ACC if c_acc is None else c_acc
    c_gdn = C_GDN if c_gdn is None else c_gdn
    u = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11, "fp32": 0.0}[out_fmt]
    a = ref.abs()
    b = u * a + c_acc * mag + (c_gdn * a if gdn else 0.0)
    if out_fmt == "fp16":
        b = b + 2.0 ** -25                             # half the fp16 subnormal spacing
    return b


def ratio(got: torch.Tensor, r: Ref, *, act: bool = False, c_acc: float = None, c_gdn: float = None):
    """(max err / bound over the written elements, all unwritten elements unchanged).  Infinite / NaN outputs give
    an infinite ratio."""
    ref, mag, wr = (r.act_ref, r.act_mag, r.act_written) if act else (r.ref, r.mag, r.written)
    fmt = "bf16" if act else r.out_fmt
    g = got.detach().to(torch.float64)
    bnd = bound(ref, mag, fmt, r.gdn and not act, c_acc, c_gdn)
    err = (g - ref).abs()
    q = torch.where(wr & (err > 0), err / bnd, torch.zeros_like(err))      # exact zeros pass a zero bound
    q = torch.where(wr & ~torch.isfinite(g), torch.full_like(q, float("inf")), q)
    untouched = bool(torch.equal(torch.where(wr, torch.zeros_like(g), g), torch.where(wr, torch.zeros_like(ref), ref)))
    return float(q.max()) if bool(wr.any()) else 0.0, untouched


def old_bar_accepts(got: torch.Tensor, r: Ref) -> bool:
    """tools/conv_diag.run_case's bar: max|got - ref| <= k * max|ref| over the written channels (bf16 output: k =
    1.2e-2, 3e-2 with GDN; fp16: 1.5e-3 / 4e-3; fp32 output 2e-3 (bf16) / 1e-3 (fp16))."""
    g = got.detach().to(torch.float64)
    err = float(((g - r.ref).abs() * r.written).max())
    scale = float((r.ref.abs() * r.written).max()) + 1e-9
    k = {"bf16": 3e-2 if r.gdn else 1.2e-2, "fp16": 4e-3 if r.gdn else 1.5e-3, "fp32": 3e-2 if r.gdn else 2e-3}[r.out_fmt]
    return err <= k * scale
