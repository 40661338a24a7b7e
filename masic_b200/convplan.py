"""Python handle on one tensor-core conv layer (a MasicConvPlan of the C ABI).

A plan binds its input/output activation buffers (NHWC, bf16 in, bf16 or fp32 out), the
packed weights and the epilogue (bias, activation, fused GDN/IGDN, per-pixel scale) once;
`launch()` is then a single kernel launch that can be captured into a CUDA graph.

Reference call sites replaced: compressai/models/utils.py:128-146 (conv/deconv),
compressai/layers/gdn.py:77-92, compressai/layers/layers.py:75-78 (MaskedConv2d).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import (ACT_LEAKY, ACT_NONE, ACT_RELU, CONV, CONV_XFOLD4, CONV_XFOLD8, DECONV_S2, DECONV_S2_SUBPIX, FMT_BF16,
                   FMT_F16, GDN_FWD, GDN_INV, GDN_NONE, ConvDesc, act_dtype, check)

# MaskedConv2d mask 'A' for a 5x5 kernel (layers.py:68-73): rows 0-1 and (2,0),(2,1)
MASK_A_5x5 = sum(1 << (ky * 5 + kx) for ky in range(5) for kx in range(5)
                 if ky < 2 or (ky == 2 and kx < 2))


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def pack_weights(w: torch.Tensor, kind: int, transposed: bool, ksize: int, c_in: int, c_out: int,
                 c_out_pad: int, f16: int = FMT_BF16) -> torch.Tensor:
    """fp32 torch-layout weights -> 16-bit [k-block][c_out_pad][64] (device), bf16 or fp16."""
    lib = _lib.load()
    w = w.detach().to(torch.float32).contiguous()
    nbytes = lib.masic_packed_weight_bytes(kind, ksize, c_in, c_out_pad)
    dst = torch.empty(nbytes // 2, dtype=act_dtype(f16), device=w.device)
    check(lib.masic_pack_conv_weights(w.data_ptr(), kind, int(transposed), ksize, c_in, c_out,
                                      c_out_pad, dst.data_ptr(), int(f16), _stream()), "masic_pack_conv_weights")
    return dst


def gdn_prepare(beta: torch.Tensor, gamma: torch.Tensor, beta_min: float = 1e-6, f16: int = FMT_BF16):
    """Stored (re-parametrised) beta/gamma -> effective beta' (fp32), gamma' (fp32, and 16-bit in the given format)."""
    lib = _lib.load()
    c = beta.numel()
    beta = beta.detach().float().contiguous()
    gamma = gamma.detach().float().contiguous()
    b = torch.empty(c, dtype=torch.float32, device=beta.device)
    g32 = torch.empty(c, c, dtype=torch.float32, device=beta.device)
    g16 = torch.empty(c, c, dtype=act_dtype(f16), device=beta.device)
    check(lib.masic_gdn_prepare(beta.data_ptr(), gamma.data_ptr(), c, float(beta_min), b.data_ptr(),
                                g32.data_ptr(), g16.data_ptr(), int(f16), _stream()), "masic_gdn_prepare")
    return b, g32, g16


class PackedConv:
    """Weights of one conv layer in the form the tensor-core kernel reads: bf16 k-blocks,
    zero-padded fp32 bias, re-parametrised GDN beta' / bf16 gamma'.  Shared by every plan
    that runs the layer (encoder1 runs twice per stereo pair, MASIC.py:746,822)."""

    def __init__(self, *, kind: int = CONV, ksize: int, c_in: int, c_out: int, n_tile: int,
                 weight: torch.Tensor, transposed: bool = False, bias: Optional[torch.Tensor] = None,
                 c_out_pad: Optional[int] = None, gdn: int = GDN_NONE,
                 gdn_beta: Optional[torch.Tensor] = None, gdn_gamma: Optional[torch.Tensor] = None,
                 f16: int = FMT_BF16):
        self.kind, self.ksize, self.c_in, self.c_out, self.n_tile = kind, ksize, c_in, c_out, n_tile
        self.transposed, self.gdn, self.f16 = transposed, gdn, int(f16)
        self.eff_out = 4 * c_out if kind == DECONV_S2_SUBPIX else c_out
        self.c_out_pad = c_out_pad if c_out_pad is not None else -(-self.eff_out // n_tile) * n_tile
        dev = weight.device
        pack_cin = weight.shape[1] if kind in (CONV_XFOLD4, CONV_XFOLD8) else c_in     # XFOLD: real channels of w
        self.w_packed = pack_weights(weight, kind, transposed, ksize, pack_cin, c_out, self.c_out_pad, self.f16)
        self.bias = None
        if bias is not None:
            b = torch.zeros(self.c_out_pad, dtype=torch.float32, device=dev)
            if kind == DECONV_S2_SUBPIX:
                b[:4 * c_out] = bias.detach().float().repeat(4)
            else:
                b[:c_out] = bias.detach().float()
            self.bias = b
        self.beta = self.gamma16 = None
        if gdn != GDN_NONE:
            # the norm MMA of the fused GDN runs on bf16 operands in both formats (conv_tc.cu: pack_norm_operand)
            self.beta, _, self.gamma16 = gdn_prepare(gdn_beta, gdn_gamma, f16=FMT_BF16)

    def repack(self, weight: torch.Tensor, bias: Optional[torch.Tensor] = None) -> None:
        """Re-pack changed weights IN PLACE (same device buffers, so bound plans stay valid): the training step
        calls this after every optimizer step."""
        lib = _lib.load()
        w = weight.detach()
        if w.dtype != torch.float32 or not w.is_contiguous():
            w = w.float().contiguous()
        pack_cin = w.shape[1] if self.kind in (CONV_XFOLD4, CONV_XFOLD8) else self.c_in
        check(lib.masic_pack_conv_weights(w.data_ptr(), self.kind, int(self.transposed), self.ksize, pack_cin,
                                          self.c_out, self.c_out_pad, self.w_packed.data_ptr(), self.f16, _stream()),
              "masic_pack_conv_weights")
        self._keep = w
        if bias is not None and self.bias is not None:
            if self.kind == DECONV_S2_SUBPIX:
                self.bias[:4 * self.c_out].copy_(bias.detach().float().repeat(4))
            else:
                self.bias[:self.c_out].copy_(bias.detach().float())


class PackBatch:
    """Every (PackedConv, weight, bias) re-pack of a training step as one kernel launch (masic_pack_batch_*).  The
    weights / biases must be fp32 contiguous tensors whose storage stays put (nn.Parameters updated in place)."""

    def __init__(self, jobs: Sequence[Tuple["PackedConv", torch.Tensor, Optional[torch.Tensor]]]):
        lib = _lib.load()
        arr = (_lib.PackJob * len(jobs))()
        self._keep = []
        for a, (pk, w, b) in zip(arr, jobs):
            assert w.dtype == torch.float32 and w.is_contiguous() and w.is_cuda, "PackBatch needs fp32 contiguous weights"
            assert pk.f16 == FMT_BF16, "PackBatch re-packs bf16 weights (the training step's format)"
            a.w, a.dst = w.data_ptr(), pk.w_packed.data_ptr()
            if b is not None and pk.bias is not None:
                assert b.dtype == torch.float32 and b.is_contiguous()
                a.bias_src, a.bias_dst = b.data_ptr(), pk.bias.data_ptr()
            a.kind, a.transposed, a.ksize = pk.kind, int(pk.transposed), pk.ksize
            a.c_in = w.shape[1] if pk.kind in (CONV_XFOLD4, CONV_XFOLD8) else pk.c_in
            a.c_out, a.c_out_pad = pk.c_out, pk.c_out_pad
            self._keep.append((pk, w, b))
        h = C.c_void_p()
        check(lib.masic_pack_batch_create(arr, len(jobs), C.byref(h)), "masic_pack_batch_create")
        self._h, self._lib, self.n_jobs = h, lib, len(jobs)

    def launch(self, stream: Optional[int] = None) -> None:
        check(self._lib.masic_pack_batch_launch(self._h, _stream() if stream is None else stream),
              "masic_pack_batch_launch")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.masic_pack_batch_destroy(h)
            self._h = None


class ConvPlan:
    def __init__(self, *, packed: Optional[PackedConv] = None, kind: int = CONV, ksize: int = 0,
                 stride: int = 1, tap_mask: int = 0,
                 x: torch.Tensor, in_coff: int = 0, c_in: int = 0,
                 weight: Optional[torch.Tensor] = None, transposed: bool = False,
                 bias: Optional[torch.Tensor] = None,
                 c_out: int = 0, n_tile: int = 0, c_out_pad: Optional[int] = None,
                 out: torch.Tensor, out_coff: int = 0,
                 act: int | Sequence[int] = ACT_NONE,
                 gdn: int = GDN_NONE, gdn_beta: Optional[torch.Tensor] = None,
                 gdn_gamma: Optional[torch.Tensor] = None,
                 rowscale: Optional[torch.Tensor] = None, rs_off: int = 0,
                 residual0: Optional[torch.Tensor] = None, res0_coff: int = 0,
                 residual1: Optional[torch.Tensor] = None, res1_coff: int = 0,
                 nt_in_coff: Optional[Sequence[int]] = None, nt_out_coff: Optional[Sequence[int]] = None,
                 nt_out_img: Optional[Sequence[int]] = None, cta_pairs: bool = False, pdl: bool = False,
                 w_in: Optional[int] = None, out_blk_images: bool = False,
                 act_out: Optional[torch.Tensor] = None, act_out_coff: int = 0):
        """act_out (training, with residual0): bf16 buffer that also receives act(conv + bias) before the residual
        adds, at channel act_out_coff (masic_conv_plan_set_act_out)."""
        lib = _lib.load()
        assert x.is_cuda and x.dtype in (torch.bfloat16, torch.float16) and x.dim() == 4 and x.is_contiguous()
        assert out.is_cuda and out.dim() == 4 and out.is_contiguous()
        if packed is None:      # the format follows the input buffer
            packed = PackedConv(kind=kind, ksize=ksize, c_in=c_in, c_out=c_out, n_tile=n_tile, weight=weight,
                                transposed=transposed, bias=bias, c_out_pad=c_out_pad, gdn=gdn,
                                gdn_beta=gdn_beta, gdn_gamma=gdn_gamma,
                                f16=FMT_F16 if x.dtype == torch.float16 else FMT_BF16)
        self.packed = packed
        fmt = act_dtype(packed.f16)
        assert x.dtype == fmt, f"input buffer is {x.dtype}, the packed weights are {fmt}"
        assert out.dtype in (fmt, torch.float32), f"output buffer is {out.dtype}, expected {fmt} or float32"
        w_logical = w_in
        n, h_in, w_in, in_cp = x.shape
        if packed.kind in (CONV_XFOLD4, CONV_XFOLD8):          # padded image rows: [N][H][W + IMG_XPAD][16 or 8]
            w_in -= _lib.IMG_XPAD
        if w_logical is not None:                              # rows wider than the logical image (MasicConvDesc.in_row_pixels)
            assert w_logical <= w_in
            row_pixels, w_in = w_in, w_logical
        else:
            row_pixels = 0
        self.rowscale = rowscale
        self.x, self.out = x, out       # keep the bound buffers alive

        d = ConvDesc()
        d.kind, d.ksize, d.stride, d.tap_mask = packed.kind, packed.ksize, stride, tap_mask
        d.n, d.h_in, d.w_in = n, h_in, w_in
        d.c_in, d.c_out, d.c_out_pad, d.n_tile = packed.c_in, packed.eff_out, packed.c_out_pad, packed.n_tile
        d.in_, d.in_cpitch, d.in_coff = x.data_ptr(), in_cp, in_coff
        d.w_packed = packed.w_packed.data_ptr()
        d.bias = _ptr(packed.bias)
        d.out, d.out_cpitch, d.out_coff = out.data_ptr(), out.shape[3], out_coff
        d.out_fp32 = int(out.dtype == torch.float32)
        n_nt = packed.c_out_pad // packed.n_tile
        acts = [act] * n_nt if isinstance(act, int) else list(act)
        assert len(acts) == n_nt, (len(acts), n_nt)
        for i, a in enumerate(acts):
            d.act[i] = a
        d.gdn = packed.gdn
        d.gamma_packed, d.beta = _ptr(packed.gamma16), _ptr(packed.beta)
        if rowscale is not None:
            assert rowscale.dtype == torch.float32 and rowscale.is_contiguous() and rowscale.dim() == 4
            d.rowscale, d.rs_stride, d.rs_off = rowscale.data_ptr(), rowscale.shape[3], rs_off
        for i, (r, off) in enumerate(((residual0, res0_coff), (residual1, res1_coff))):
            if r is not None:
                assert r.is_cuda and r.dtype == fmt and r.dim() == 4 and r.is_contiguous()
                assert r.shape[:3] == out.shape[:3], (r.shape, out.shape)
                setattr(d, f"residual{i}", r.data_ptr())
                setattr(d, f"res{i}_cpitch", r.shape[3])
                setattr(d, f"res{i}_coff", off)
        self.residuals = (residual0, residual1)
        if nt_in_coff is not None or nt_out_coff is not None or nt_out_img is not None:   # grouped launch
            tabs = []
            for name, tab, default in (("nt_in_coff", nt_in_coff, [0] * n_nt),
                                       ("nt_out_coff", nt_out_coff, [i * packed.n_tile for i in range(n_nt)]),
                                       ("nt_out_img", nt_out_img, [0] * n_nt)):
                tab = list(default if tab is None else tab)
                assert len(tab) == n_nt, (name, len(tab), n_nt)
                arr = (C.c_int * n_nt)(*tab)
                tabs.append(arr)
                setattr(d, name, C.cast(arr, C.POINTER(C.c_int)))
            self._tabs = tabs
            d.out_images = out.shape[0]
        elif not out_blk_images:
            assert out.shape[0] == n, (out.shape, n)
        d.cta_pairs = int(cta_pairs)
        d.f16 = packed.f16
        d.pdl = int(pdl)
        d.in_row_pixels = int(row_pixels)
        d.out_blk_images = int(out_blk_images)
        self._desc = d
        handle = C.c_void_p()
        check(lib.masic_conv_plan_create(C.byref(d), C.byref(handle)), "masic_conv_plan_create")
        self._h = handle
        self._lib = lib
        self.act_out = act_out
        if act_out is not None:
            assert act_out.is_cuda and act_out.dtype == torch.bfloat16 and act_out.is_contiguous()
            assert act_out.shape[:3] == out.shape[:3], (act_out.shape, out.shape)
            check(lib.masic_conv_plan_set_act_out(handle, act_out.data_ptr(), act_out.shape[3], act_out_coff),
                  "masic_conv_plan_set_act_out")
        fl, by, nw, sm = C.c_double(), C.c_double(), C.c_int(), C.c_int()
        lib.masic_conv_plan_info(handle, C.byref(fl), C.byref(by), C.byref(nw), C.byref(sm))
        self.flops, self.hbm_bytes, self.work_items, self.smem_bytes = fl.value, by.value, nw.value, sm.value

    @property
    def c_out_pad(self) -> int:
        return self.packed.c_out_pad

    def launch(self, stream: Optional[int] = None) -> None:
        check(self._lib.masic_conv_plan_launch(self._h, _stream() if stream is None else stream),
              "masic_conv_plan_launch")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.masic_conv_plan_destroy(h)
            self._h = None


def fold8_weights_5x5_s1(weight: torch.Tensor, bias: Optional[torch.Tensor], transposed: bool,
                         slots: Optional[Sequence[int]] = None):
    """A 5x5 stride-1 pad-2 layer with <= 8 input and 3 output channels (after_conv, MASIC.py:600,616) as a conv over
    PIXEL-FOLDED data: the NHWC pitch-8 image [H][W + IMG_XPAD][8] (pixel x at column x + IMG_XOFF = 2) is read as
    [H][(W + 8) / 8][64] — one "pixel" = 8 image pixels x 8 channels — and output block xb (image pixels 8 xb .. 8 xb + 7)
    needs blocks xb and xb + 1 only, i.e. taps kx' = 2, 3 of a 5-wide kernel.  Returns the (48, 64, 5, 5) weight
    (row co * 16 + j = output channel co of pixel j, j < 8; column p * 8 + c = channel c of the block's pixel p), the
    48-entry bias and the tap mask (10 live taps).  With MasicConvDesc.out_blk_images the three 16-column blocks land in
    the three planes of an NCHW tensor.  slots[ci] = position of input channel ci inside the 8-channel pixel
    (default 0, 1, 2, ...)."""
    dev = weight.device
    w = weight.detach().float().cpu()                                     # ~1000 tiny slice copies: on the host
    wc = w.flip(2, 3).permute(1, 0, 2, 3) if transposed else w           # correlation kernel (c_out, c_in, 5, 5)
    c_out, c_in = wc.shape[0], wc.shape[1]
    assert c_out == 3 and c_in <= 8 and tuple(wc.shape[2:]) == (5, 5)
    big = torch.zeros(48, 64, 5, 5, dtype=torch.float32)
    slots = list(range(c_in)) if slots is None else list(slots)
    assert len(slots) == c_in and len(set(slots)) == c_in and all(0 <= t < 8 for t in slots)
    for kxp, base in ((2, 0), (3, 8)):
        for pq in range(8):
            q = base + pq                       # column offset inside the 16-pixel window: image pixel 8 xb - 2 + q
            for j in range(8):
                kx = q - j                      # output pixel 8 xb + j reads image pixel 8 xb + j + kx - 2
                if 0 <= kx < 5:
                    for co in range(3):
                        for ci, sl in enumerate(slots):
                            big[co * 16 + j, pq * 8 + sl, :, kxp] = wc[co, ci, :, kx]
    b48 = torch.zeros(48, dtype=torch.float32)
    if bias is not None:
        bh = bias.detach().float().cpu()
        for co in range(3):
            b48[co * 16:co * 16 + 8] = bh[co]
    mask = 0
    for ky in range(5):
        mask |= (1 << (ky * 5 + 2)) | (1 << (ky * 5 + 3))
    return big.to(dev), b48.to(dev), mask


class DeconvImgPlan:
    """g_s_conv4 — ConvTranspose2d(128, 3, k=5, s=2, p=2, op=1) at image resolution (MasicDeconvImgPlan of the C ABI,
    csrc/deconv_img.cu): NHWC 16-bit (n, h, w, 128) in, NCHW fp32 (n, 3, 2h, 2w) out, optional after_gdn (IGDN over the
    three channels) fused.  `weight` is the module's (128, 3, 5, 5) tensor."""

    def __init__(self, *, x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor],
                 out: Optional[torch.Tensor], igdn_beta: Optional[torch.Tensor] = None,
                 igdn_gamma: Optional[torch.Tensor] = None, out16: Optional[torch.Tensor] = None, out16_coff: int = 0,
                 out16_xoff: int = 0):
        """out16: optional (n, 2h, row_pixels, pitch) 16-bit NHWC image that receives the 3 channels at channel
        out16_coff of column x + out16_xoff (`out` may then be None)."""
        import numpy as np
        lib = _lib.load()
        assert x.is_cuda and x.dtype in (torch.bfloat16, torch.float16) and x.dim() == 4 and x.is_contiguous()
        n, h, w, cp = x.shape
        assert cp == 128 and tuple(weight.shape) == (128, 3, 5, 5), (x.shape, weight.shape)
        assert out is not None or out16 is not None
        if out is not None:
            assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (n, 3, 2 * h, 2 * w)
        f16 = int(x.dtype == torch.float16)
        self.w_packed = torch.empty(lib.masic_deconv_img_weight_bytes() // 2, dtype=x.dtype, device=x.device)
        wt = weight.detach().float().contiguous()
        check(lib.masic_deconv_img_pack_weights(wt.data_ptr(), self.w_packed.data_ptr(), f16, _stream()),
              "masic_deconv_img_pack_weights")
        self.bias = None if bias is None else bias.detach().float().contiguous()
        gdn, pb, pg = GDN_NONE, None, None
        if igdn_beta is not None:
            gdn = GDN_INV
            self._b = np.ascontiguousarray(igdn_beta.detach().float().cpu().numpy())
            self._g = np.ascontiguousarray(igdn_gamma.detach().float().cpu().numpy())
            pb, pg = self._b.ctypes.data, self._g.ctypes.data
        self.x, self.out = x, out
        hdl = C.c_void_p()
        check(lib.masic_deconv_img_plan_create(x.data_ptr(), n, h, w, cp, self.w_packed.data_ptr(), _ptr(self.bias), gdn,
                                               pb, pg, _ptr(out), f16, C.byref(hdl)), "masic_deconv_img_plan_create")
        self._h, self._lib = hdl, lib
        self.out16 = out16
        if out16 is not None:
            assert out16.is_cuda and out16.dtype in (torch.bfloat16, torch.float16) and out16.is_contiguous()
            assert out16.dim() == 4 and out16.shape[0] == n and out16.shape[1] == 2 * h
            check(lib.masic_deconv_img_plan_set_out16(hdl, out16.data_ptr(), out16.shape[3], out16.shape[2], out16_xoff,
                                                      out16_coff, int(out16.dtype == torch.float16)),
                  "masic_deconv_img_plan_set_out16")
        self.flops = 2.0 * n * h * w * 128 * 75
        self.work_items = n * (-(-w // 14)) * (h // 8)
        self.smem_bytes = 0
        self.hbm_bytes = n * h * w * (256.0 + (48.0 if out is not None else 0.0) + (24.0 if out16 is not None else 0.0))

    def launch(self, stream: Optional[int] = None) -> None:
        check(self._lib.masic_deconv_img_plan_launch(self._h, _stream() if stream is None else stream),
              "masic_deconv_img_plan_launch")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.masic_deconv_img_plan_destroy(h)
            self._h = None


class WgradPlan:
    """Tensor-core weight gradient of one conv / transposed-conv layer (MasicWgradPlan of the C ABI).
    `lo` / `hi` are the bound NHWC bf16 buffers (see include/masic_b200.h), `dw` the fp32 torch-layout gradient."""

    # Partial-sum workspace: plans of one device share the current buffer while it is large enough; a plan that needs
    # more allocates a new one for itself and its successors.  Every plan keeps a reference to the buffer it bound,
    # so a CUDA graph that captured an earlier plan's launch never sees its workspace freed (ADVICE r1).
    _ws: dict = {}

    def __init__(self, *, ksize: int, stride: int, lo: torch.Tensor, c_lo: int, hi: torch.Tensor, c_hi: int,
                 dw: torch.Tensor, lo_coff: int = 0, hi_coff: int = 0, tap_mask: int = 0, accumulate: bool = False):
        lib = _lib.load()
        for t in (lo, hi):
            assert t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 4 and t.is_contiguous()
        assert dw.is_cuda and dw.dtype == torch.float32 and dw.is_contiguous()
        n, h_lo, w_lo, lo_cp = lo.shape
        assert hi.shape[0] == n and hi.shape[1] == h_lo * stride and hi.shape[2] == w_lo * stride, (lo.shape, hi.shape)
        d = _lib.WgradDesc()
        d.ksize, d.stride, d.tap_mask = ksize, stride, tap_mask
        d.n, d.h_lo, d.w_lo = n, h_lo, w_lo
        d.lo, d.lo_cpitch, d.lo_coff, d.c_lo = lo.data_ptr(), lo_cp, lo_coff, c_lo
        d.hi, d.hi_cpitch, d.hi_coff, d.c_hi = hi.data_ptr(), hi.shape[3], hi_coff, c_hi
        d.dw, d.accumulate = dw.data_ptr(), int(accumulate)
        self._desc, self.lo, self.hi, self.dw = d, lo, hi, dw
        h = C.c_void_p()
        check(lib.masic_wgrad_plan_create(C.byref(d), C.byref(h)), "masic_wgrad_plan_create")
        self._h, self._lib = h, lib
        fl, nc = C.c_double(), C.c_int()
        lib.masic_wgrad_plan_info(h, C.byref(fl), C.byref(nc))
        self.flops, self.n_ctas = fl.value, nc.value
        need = lib.masic_wgrad_plan_workspace_bytes(h)
        key = lo.device.index
        cur = WgradPlan._ws.get(key)
        if cur is None or cur.numel() * 4 < need:
            WgradPlan._ws[key] = torch.empty(need // 4 + 1024, dtype=torch.float32, device=lo.device)
        self._bound_ws = WgradPlan._ws[key]

    def launch(self, stream: Optional[int] = None) -> None:
        ws = self._bound_ws
        check(self._lib.masic_wgrad_plan_launch(self._h, ws.data_ptr(), _stream() if stream is None else stream),
              "masic_wgrad_plan_launch")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.masic_wgrad_plan_destroy(h)
            self._h = None


def conv_direct(x: torch.Tensor, c_in: int, weight: torch.Tensor, *, transposed: bool, ksize: int,
                stride: int, tap_mask: int = 0, bias: Optional[torch.Tensor] = None,
                in_coff: int = 0, round_w_bf16: bool = True) -> torch.Tensor:
    """CUDA-core direct conv over NHWC bf16 input -> NHWC fp32 (on-device cross-check)."""
    lib = _lib.load()
    n, h, w, cp = x.shape
    c_out = weight.shape[1] if transposed else weight.shape[0]
    ho, wo = (h * stride, w * stride) if transposed else (-(-h // stride), -(-w // stride))
    out = torch.empty(n, ho, wo, c_out, dtype=torch.float32, device=x.device)
    wt = weight.detach().float().contiguous()
    bt = None if bias is None else bias.detach().float().contiguous()
    check(lib.masic_conv_direct_nhwc(x.data_ptr(), n, h, w, cp, in_coff, c_in, wt.data_ptr(),
                                     int(transposed), ksize, stride, tap_mask, _ptr(bt), c_out,
                                     out.data_ptr(), c_out, 0, int(round_w_bf16), int(x.dtype == torch.float16), _stream()),
          "masic_conv_direct_nhwc")
    return out
