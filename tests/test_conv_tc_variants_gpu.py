"""Every instantiation of conv_tc_kernel<CG2, EPI, F16> against the float64 reference of tests/conv_ref.py, per element.

The module derives from each case's descriptor which of the 15 instantiations it selects (the rule of
masic_conv_plan_create / masic_conv_plan_launch) and test_all_instantiations_covered asserts that the cases reach all
15.  Each case compares the whole output buffer: computed elements within conv_ref.bound, every other element still
holding the sentinel.  Each prints one JSON line {"case", "inst", "max_err_over_bound"}.

Axes: 1, 2 and 3 spatial tiles; an odd tile count with several n-tiles (CTA-pair items cut at n-tile boundaries); more
than 2 x 148 items; ragged h / w and w < 8; batches of 1 and 3; n_tile 16 ... 256 in the plain epilogue with 16-bit and
fp32 output, and every n_tile CTA pairs accept; mixed per-n-tile activations; rowscale with rs_stride 3 and rs_off 0..2;
one and two residuals at channel offsets; grouped tables; out_coff inside a wider buffer; garbage in unread input
channels; fp16 saturation; in_row_pixels and out_blk_images; PDL chains in a CUDA graph; bit-identity of repeated
launches, graph replay, batch slicing and CTA pairs on / off.
"""
from __future__ import annotations

import json

import pytest
import torch

import conv_ref as R

pytestmark = pytest.mark.gpu

PLAIN, GDN, RES, GDN2, RESA = "PLAIN", "GDN", "RES", "GDN2", "RESA"
ALL_INSTANTIATIONS = ({(c, e, f) for c in (0, 1) for e in (PLAIN, GDN, RES) for f in ("bf16", "fp16")}
                      | {(0, GDN2, "bf16"), (0, GDN2, "fp16"), (0, RESA, "bf16")})
MASK_A_5x5 = sum(1 << (ky * 5 + kx) for ky in range(5) for kx in range(5) if ky < 2 or (ky == 2 and kx < 2))
SENTINEL = 777.0


def instantiation(c: dict, fmt: str):
    """(CG2, EPI, format) that masic_conv_plan_launch picks for case `c`."""
    kind, k = c.get("kind", R.CONV), c["k"]
    cg2 = int(bool(c.get("pairs")))
    if c.get("gdn"):
        n_var = 4 if kind == R.DECONV_S2 else 1
        if kind == R.CONV_XFOLD4:
            bops = 10
        elif kind == R.CONV_XFOLD8:
            bops = 5
        else:
            live = bin(c.get("tap_mask", 0)).count("1") or (9 if kind == R.DECONV_S2_SUBPIX else k * k)
            bops = live * -(-c["c_in"] // 64)
        epi = GDN2 if (not cg2 and n_var == 1 and bops <= 6) else GDN
    elif c.get("act_out"):
        epi = RESA
    elif c.get("res"):
        epi = RES
    else:
        epi = PLAIN
    return cg2, epi, fmt


# ---------------------------------------------------------------------------------------------------- the matrix
def _nt_case(nt, pairs, fp32):
    return dict(k=3, n=1, h=21, w=19, c_in=64, c_out=2 * nt - 16, n_tile=nt, act=R.ACT_LEAKY, out_fp32=fp32,
                pairs=pairs, out_coff=8, out_extra=8)


CASES = {
    # tile-walk edges
    "tiles1": dict(k=3, n=1, h=16, w=8, c_in=64, c_out=64, n_tile=64),
    "tiles2_ragged": dict(k=3, n=1, h=13, w=11, c_in=64, c_out=64, n_tile=64, act=R.ACT_RELU),
    "tiles3_w5_batch3": dict(k=3, n=3, h=10, w=5, c_in=64, c_out=96, n_tile=96),
    "tiles1_pairs": dict(k=3, n=1, h=16, w=8, c_in=64, c_out=64, n_tile=64, pairs=True),
    "tiles2_pairs": dict(k=3, n=1, h=13, w=11, c_in=64, c_out=64, n_tile=64, pairs=True),
    "tiles3_w5_batch3_pairs": dict(k=3, n=3, h=10, w=5, c_in=64, c_out=96, n_tile=96, pairs=True),
    "odd_tiles_4nt": dict(k=1, n=1, h=40, w=24, c_in=128, c_out=256, n_tile=64,
                          act=[R.ACT_RELU, R.ACT_LEAKY, R.ACT_NONE, R.ACT_LEAKY]),
    "odd_tiles_4nt_pairs": dict(k=1, n=1, h=40, w=24, c_in=128, c_out=256, n_tile=64, pairs=True,
                                act=[R.ACT_RELU, R.ACT_LEAKY, R.ACT_NONE, R.ACT_LEAKY]),
    "many_items": dict(k=1, n=3, h=190, w=190, c_in=64, c_out=256, n_tile=128),
    "many_items_pairs": dict(k=1, n=3, h=190, w=190, c_in=64, c_out=256, n_tile=128, pairs=True),
    "gmm_l0_18nt_pairs": dict(k=1, n=1, h=19, w=34, c_in=320, c_out=3456, n_tile=192, pairs=True,
                              act=[R.ACT_RELU] * 6 + [R.ACT_LEAKY] * 12),
    # strided / transposed / masked / sub-pixel
    "s2_5x5": dict(k=5, stride=2, n=1, h=38, w=36, c_in=128, c_out=192, n_tile=192, out_fp32=True),
    "s2_5x5_pairs": dict(k=5, stride=2, n=3, h=34, w=18, c_in=128, c_out=128, n_tile=128, pairs=True),
    "deconv_leaky": dict(kind=R.DECONV_S2, k=5, n=1, h=11, w=9, c_in=128, c_out=288, n_tile=192, act=R.ACT_LEAKY),
    "deconv_pairs": dict(kind=R.DECONV_S2, k=5, n=1, h=11, w=9, c_in=128, c_out=192, n_tile=192, pairs=True,
                         act=R.ACT_LEAKY),
    "subpix_fp32": dict(kind=R.DECONV_S2_SUBPIX, k=5, n=1, h=24, w=13, c_in=128, c_out=3, n_tile=16, out_fp32=True),
    "masked5x5_rs1_pairs": dict(k=5, tap_mask=MASK_A_5x5, n=1, h=20, w=13, c_in=192, c_out=384, n_tile=192,
                                pairs=True, rowscale=True, rs_off=1, out_coff=384, out_extra=0),
    "k1_transposed": dict(k=1, n=1, h=16, w=9, c_in=128, c_out=256, n_tile=128, transposed=True),
    # epilogue inputs
    "rowscale_rs0": dict(k=3, n=2, h=21, w=13, c_in=64, c_out=96, n_tile=96, rowscale=True, rs_off=0),
    "rowscale_rs1": dict(k=3, n=2, h=21, w=13, c_in=64, c_out=96, n_tile=96, rowscale=True, rs_off=1,
                         act=R.ACT_LEAKY),
    "rowscale_rs2_pairs": dict(k=3, n=2, h=21, w=13, c_in=64, c_out=96, n_tile=96, rowscale=True, rs_off=2,
                               pairs=True),
    "res1": dict(k=3, n=2, h=19, w=13, c_in=64, c_out=64, n_tile=64, act=R.ACT_LEAKY, res=1, out_coff=16, out_extra=0),
    "res2": dict(k=3, n=1, h=19, w=13, c_in=96, c_out=96, n_tile=96, act=R.ACT_LEAKY, res=2, out_coff=16, out_extra=16),
    "res2_rowscale": dict(k=3, n=1, h=19, w=13, c_in=64, c_out=128, n_tile=64, act=R.ACT_LEAKY, res=2, rowscale=True,
                          rs_off=2),
    "res1_pairs": dict(k=3, n=2, h=19, w=13, c_in=64, c_out=64, n_tile=64, act=R.ACT_LEAKY, res=1, pairs=True),
    "res2_pairs": dict(k=3, n=1, h=19, w=13, c_in=128, c_out=192, n_tile=192, act=R.ACT_LEAKY, res=2, pairs=True,
                       out_coff=16, out_extra=16),
    "resa": dict(k=3, n=2, h=19, w=13, c_in=64, c_out=64, n_tile=64, act=R.ACT_LEAKY, res=2, act_out=True,
                 formats=("bf16",)),
    "grouped": dict(k=1, n=2, h=19, w=13, c_in=128, c_out=384, n_tile=96, grouped=True),
    "grouped_pairs": dict(k=1, n=2, h=19, w=13, c_in=128, c_out=384, n_tile=96, grouped=True, pairs=True),
    "cin48_garbage": dict(k=3, n=1, h=18, w=18, c_in=48, in_cp=64, c_out=64, n_tile=64, garbage=True),
    "cin48_garbage_coff": dict(k=3, n=1, h=18, w=18, c_in=48, in_coff=16, in_cp=128, c_out=64, n_tile=64, garbage=True),
    "saturate": dict(k=1, n=1, h=16, w=16, c_in=64, c_out=64, n_tile=64, big=True),
    # fused GDN / IGDN
    "gdn_5x5s2": dict(k=5, stride=2, n=1, h=34, w=22, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_FWD),
    "gdn_5x5s2_pairs": dict(k=5, stride=2, n=3, h=34, w=22, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_FWD, pairs=True),
    "gdn_5x5s2_pairs_rs": dict(k=5, stride=2, n=1, h=34, w=22, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_FWD,
                               pairs=True, rowscale=True, rs_off=2),
    "igdn_deconv": dict(kind=R.DECONV_S2, k=5, n=1, h=9, w=11, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_INV),
    "gdn_xfold4": dict(kind=R.CONV_XFOLD4, k=5, stride=2, n=2, h=40, w=38, c_in=64, c_out=128, n_tile=128,
                       gdn=R.GDN_FWD),
    "gdn2_xfold8": dict(kind=R.CONV_XFOLD8, k=5, stride=2, n=2, h=40, w=38, c_in=64, c_out=128, n_tile=128,
                        gdn=R.GDN_FWD),
    "gdn2_1x1_rs": dict(k=1, n=1, h=21, w=27, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_FWD, rowscale=True, rs_off=1),
    "igdn2_1x1": dict(k=1, n=3, h=9, w=7, c_in=128, c_out=128, n_tile=128, gdn=R.GDN_INV),
    # wide rows / planar output
    "rowpix_3x3": dict(k=3, n=1, h=17, w=13, row_extra=5, c_in=64, c_out=64, n_tile=64),
    "rowpix_5x5": dict(k=5, n=2, h=17, w=13, row_extra=3, c_in=64, c_out=64, n_tile=64, act=R.ACT_LEAKY),
    "planar48_fp32": dict(k=5, n=2, h=17, w=13, row_extra=1, c_in=64, c_out=48, n_tile=48, out_fp32=True, blk=True,
                          out_cp=8),
    "planar96": dict(k=3, n=2, h=17, w=13, c_in=64, c_out=96, n_tile=96, blk=True, out_cp=24),
}
for _nt in (16, 32, 48, 64, 96, 128, 192, 256):
    for _fp32 in (False, True):
        CASES[f"nt{_nt}{'_fp32' if _fp32 else ''}"] = _nt_case(_nt, False, _fp32)
PAIR_N_TILES = (32, 64, 96, 128, 160, 192, 224, 256)       # every n_tile masic_conv_plan_create accepts with CTA pairs
for _nt in PAIR_N_TILES:
    for _fp32 in (False, True):
        CASES[f"nt{_nt}{'_fp32' if _fp32 else ''}_pairs"] = _nt_case(_nt, True, _fp32)


def _dt(fmt):
    return torch.float16 if fmt == "fp16" else torch.bfloat16


def build(c: dict, fmt: str, seed: int = 0, x=None, pairs=None):
    """Operands, PackedConv and ConvPlan of case `c`.  Returns (plan, reference kwargs)."""
    from masic_b200 import _lib
    from masic_b200.convplan import ConvPlan, PackedConv
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(seed)              # data
    gw = torch.Generator(device=dev).manual_seed(seed + 1000)      # parameters: independent of the batch size
    dt = _dt(fmt)
    kind, k, n, h, w = c.get("kind", R.CONV), c["k"], c["n"], c["h"], c["w"]
    c_in, c_out, nt = c["c_in"], c["c_out"], c["n_tile"]
    stride = c.get("stride", 1)
    tr = c.get("transposed", kind in (R.DECONV_S2, R.DECONV_S2_SUBPIX))
    xfold = kind in (R.CONV_XFOLD4, R.CONV_XFOLD8)
    if x is None:
        if xfold:
            cp = 16 if kind == R.CONV_XFOLD4 else 8
            x = torch.zeros(n, h, w + _lib.IMG_XPAD, cp, device=dev)
            x[:, :, _lib.IMG_XOFF:_lib.IMG_XOFF + w, :3] = torch.rand(n, h, w, 3, device=dev, generator=g)
            x = x.to(dt)
        else:
            in_cp = c.get("in_cp", c.get("in_coff", 0) + c_in)
            x = torch.randn(n, h, w + c.get("row_extra", 0), in_cp, device=dev, generator=g)
            if c.get("garbage"):        # finite garbage in the channels up to the next 64-channel boundary
                x[..., c.get("in_coff", 0) + c_in:] = 3e3 * torch.sign(x[..., c.get("in_coff", 0) + c_in:])
            x = x.to(dt)
    if xfold:
        wt = torch.randn(c_out, 3, 5, 5, device=dev, generator=gw) / 75 ** 0.5
    else:
        fan = c_in * k * k if kind == R.CONV else c_in * 25 / 4
        wt = torch.randn(*((c_in, c_out, k, k) if tr else (c_out, c_in, k, k)), device=dev, generator=gw) / fan ** 0.5
    if c.get("big"):
        wt = wt * 3e4
    b = torch.randn(c_out, device=dev, generator=gw) * 0.1
    gb = gg = None
    if c.get("gdn"):
        gb = torch.sqrt(torch.rand(c_out, device=dev, generator=gw) * 0.5 + 0.75)
        gg = torch.sqrt(torch.rand(c_out, c_out, device=dev, generator=gw) * 0.02 + 0.1 * torch.eye(c_out, device=dev))
    f16 = int(fmt == "fp16")
    pk = PackedConv(kind=kind, ksize=k, c_in=c_in, c_out=c_out, n_tile=nt, weight=wt, transposed=tr, bias=b,
                    gdn=c.get("gdn", 0), gdn_beta=gb, gdn_gamma=gg, f16=f16)
    if kind == R.DECONV_S2:
        ho, wo = 2 * h, 2 * w
    elif stride == 2 or xfold:
        ho, wo = h // 2, w // 2
    else:
        ho, wo = h, w
    n_nt = pk.c_out_pad // nt
    out_coff = c.get("out_coff", 0)
    odt = torch.float32 if c.get("out_fp32") else dt
    kw = dict(stride=stride, tap_mask=c.get("tap_mask", 0), x=x, in_coff=c.get("in_coff", 0), act=c.get("act", 0),
              out_coff=out_coff)
    if c.get("grouped"):
        kw.update(nt_in_coff=[0, 0, 64, 64][:n_nt], nt_out_coff=[0, nt, 0, 0][:n_nt], nt_out_img=[0, 0, n, 2 * n][:n_nt])
        kw["x"] = x = torch.randn(n, h, w, 192, device=dev, generator=g).to(dt)
        out = torch.full((3 * n, ho, wo, out_coff + 2 * nt + 8), SENTINEL, device=dev, dtype=odt)
    elif c.get("blk"):
        nblk = nt // R.blk_channels(nt, odt == torch.float32)
        out = torch.full((n * nblk, ho, wo, c["out_cp"]), SENTINEL, device=dev, dtype=odt)
        kw.update(out_blk_images=True)
    else:
        out = torch.full((n, ho, wo, out_coff + pk.c_out_pad + c.get("out_extra", 0)), SENTINEL, device=dev, dtype=odt)
    kw["out"] = out
    if c.get("row_extra"):
        kw["w_in"] = w
    if c.get("rowscale"):
        kw.update(rowscale=torch.rand(n, ho, wo, 3, device=dev, generator=g) + 0.5, rs_off=c["rs_off"])
    if c.get("res"):
        kw.update(residual0=torch.randn(n, ho, wo, pk.c_out_pad + 24, device=dev, generator=g).to(dt), res0_coff=24)
        if c["res"] == 2:
            kw.update(residual1=torch.randn(n, ho, wo, pk.c_out_pad + 8, device=dev, generator=g).to(dt), res1_coff=8)
    if c.get("act_out"):
        kw.update(act_out=torch.full((n, ho, wo, pk.c_out_pad + 16), SENTINEL, device=dev, dtype=torch.bfloat16),
                  act_out_coff=16)
    pairs = c.get("pairs", False) if pairs is None else pairs
    plan = ConvPlan(packed=pk, cta_pairs=pairs, **kw)
    rkw = dict(kw, kind=kind, ksize=k, c_in=c_in, c_out=c_out, n_tile=nt, c_out_pad=pk.c_out_pad, transposed=tr,
               weight=wt, bias=b, gdn=pk.gdn, beta_p=pk.beta, gamma_p=pk.gamma16)
    return plan, rkw


def snapshot(rkw):
    """Copies of the buffers the plan writes, before the launch (the reference reads their previous contents)."""
    return {k: rkw[k].clone() for k in ("out", "act_out") if rkw.get(k) is not None}


def check(name, inst, rkw, before, extra=None):
    r = R.reference(**{**rkw, **before})
    q, untouched = R.ratio(rkw["out"], r)
    line = {"case": name, "inst": list(inst), "max_err_over_bound": round(q, 4)}
    if rkw.get("act_out") is not None:
        qa, ua = R.ratio(rkw["act_out"], r, act=True)
        line["act_out_max_err_over_bound"] = round(qa, 4)
        assert ua and qa <= 1.0, (name, qa)
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)
    assert untouched, f"{name}: an element outside the plan's output range changed"
    assert q <= 1.0, (name, q)
    return q


_PARAMS = [(name, fmt) for name, c in CASES.items() for fmt in c.get("formats", ("bf16", "fp16"))]


@pytest.mark.parametrize("name,fmt", _PARAMS, ids=[f"{a}-{b}" for a, b in _PARAMS])
def test_case(name, fmt):
    c = CASES[name]
    plan, rkw = build(c, fmt, seed=len(name))
    before = snapshot(rkw)
    plan.launch()
    torch.cuda.synchronize()
    check(name, instantiation(c, fmt), rkw, before, {"fmt": fmt, "work": plan.work_items})
    if c.get("big") and fmt == "fp16":        # saturating output: +-65504, never inf
        o = rkw["out"].float()
        assert bool(torch.isfinite(o).all()) and float(o.abs().max()) == R.F16_MAX


def test_all_instantiations_covered():
    got = {instantiation(c, fmt) for name, fmt in _PARAMS for c in (CASES[name],)}
    assert got == ALL_INSTANTIATIONS, sorted(ALL_INSTANTIATIONS - got)


# ---------------------------------------------------------------------------------------------------- refusals
def _tiny(fmt="bf16"):
    dev = torch.device("cuda:0")
    return torch.zeros(1, 16, 16, 64, dtype=_dt(fmt), device=dev)


@pytest.mark.parametrize("nt", [16, 48, 80, 112, 144, 176, 208, 240])
def test_pairs_refuse_n_tile(nt):
    """CTA pairs stage n_tile / 2 rows of B per CTA; n_tile values that are not multiples of 32 are refused."""
    from masic_b200 import _lib
    from masic_b200.convplan import ConvPlan, PackedConv
    x = _tiny()
    pk = PackedConv(ksize=1, c_in=64, c_out=nt, n_tile=nt, weight=torch.zeros(nt, 64, 1, 1, device=x.device))
    out = torch.zeros(1, 16, 16, nt, dtype=torch.float32, device=x.device)   # fp32: every n_tile % 16 has a layout
    ConvPlan(packed=pk, x=x, out=out)                       # the same plan without pairs is accepted
    with pytest.raises(_lib.MasicError):
        ConvPlan(packed=pk, x=x, out=out, cta_pairs=True)


def test_header_exclusions_refused():
    """in_row_pixels only for stride-1 MASIC_CONV; out_blk_images only for single-n-tile MASIC_CONV without GDN,
    residuals or grouped tables."""
    from masic_b200 import _lib
    from masic_b200.convplan import ConvPlan, PackedConv
    dev = torch.device("cuda:0")
    x = torch.zeros(1, 16, 20, 64, dtype=torch.bfloat16, device=dev)
    w3 = torch.zeros(64, 64, 3, 3, device=dev)
    with pytest.raises(_lib.MasicError):                    # in_row_pixels with stride 2
        ConvPlan(ksize=3, stride=2, x=x, c_in=64, weight=w3, c_out=64, n_tile=64, w_in=16,
                 out=torch.zeros(1, 8, 8, 64, dtype=x.dtype, device=dev))
    wd = torch.zeros(64, 64, 5, 5, device=dev)
    with pytest.raises(_lib.MasicError):                    # in_row_pixels on a transposed conv
        ConvPlan(kind=R.DECONV_S2, ksize=5, x=x, c_in=64, weight=wd, transposed=True, c_out=64, n_tile=64, w_in=16,
                 out=torch.zeros(1, 32, 32, 64, dtype=x.dtype, device=dev))
    o = torch.zeros(2, 16, 20, 8, dtype=torch.float32, device=dev)
    ConvPlan(ksize=3, x=x, c_in=64, weight=torch.zeros(32, 64, 3, 3, device=dev), c_out=32, n_tile=32, out=o,
             out_blk_images=True)                           # accepted: one n-tile of two 16-channel fp32 blocks
    with pytest.raises(_lib.MasicError):                    # planar output with two n-tiles
        ConvPlan(ksize=3, x=x, c_in=64, weight=torch.zeros(64, 64, 3, 3, device=dev), c_out=64, n_tile=32, out=o,
                 out_blk_images=True)
    with pytest.raises(_lib.MasicError):                    # planar output with a residual
        ConvPlan(ksize=3, x=x, c_in=64, weight=torch.zeros(32, 64, 3, 3, device=dev), c_out=32, n_tile=32, out=o,
                 out_blk_images=True, residual0=torch.zeros(2, 16, 20, 32, dtype=x.dtype, device=dev))
    with pytest.raises(_lib.MasicError):                    # planar output of a transposed conv
        ConvPlan(kind=R.DECONV_S2, ksize=5, x=x, c_in=64, weight=torch.zeros(64, 32, 5, 5, device=dev),
                 transposed=True, c_out=32, n_tile=32, out=torch.zeros(2, 32, 40, 8, device=dev), out_blk_images=True)


# ---------------------------------------------------------------------------------------------------- bit-identity
@pytest.mark.parametrize("name", ["odd_tiles_4nt", "gdn_5x5s2", "res2", "gdn2_xfold8"])
@pytest.mark.parametrize("pairs", [False, True])
def test_repeat_and_graph_bit_identical(name, pairs):
    c = CASES[name]
    if pairs and (c.get("kind") in (R.CONV_XFOLD8,)):
        pytest.skip("XFOLD8 with GDN runs as GDN2, which has no pair form")
    plan, rkw = build(c, "fp16", seed=3, pairs=pairs)
    out = rkw["out"]
    plan.launch()
    torch.cuda.synchronize()
    a = out.clone()
    out.fill_(SENTINEL)
    plan.launch()
    torch.cuda.synchronize()
    assert torch.equal(a, out)
    out.fill_(SENTINEL)
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(gr, stream=s):
            plan.launch()
    torch.cuda.current_stream().wait_stream(s)
    gr.replay()
    torch.cuda.synchronize()
    assert torch.equal(a, out)


@pytest.mark.parametrize("name", ["tiles3_w5_batch3", "s2_5x5_pairs", "gdn_5x5s2_pairs", "res1"])
@pytest.mark.parametrize("pairs", [False, True])
def test_batch_slice_bit_identical(name, pairs):
    """Image i of a batch of 3 equals the same image run alone."""
    c = dict(CASES[name], n=3)
    plan, rkw = build(c, "bf16", seed=4, pairs=pairs)
    plan.launch()
    torch.cuda.synchronize()
    for i in range(3):
        c1 = dict(c, n=1)
        x1 = rkw["x"][i:i + 1].clone()
        p1, r1 = build(c1, "bf16", seed=4, x=x1, pairs=pairs)
        for key in ("rowscale", "residual0", "residual1"):           # same per-pixel operands as image i
            if rkw.get(key) is not None:
                r1[key].copy_(rkw[key][i:i + 1])
        p1.launch()
        torch.cuda.synchronize()
        assert torch.equal(r1["out"], rkw["out"][i:i + 1]), (name, pairs, i)


@pytest.mark.parametrize("name", ["odd_tiles_4nt", "s2_5x5_pairs", "gdn_5x5s2", "res2", "masked5x5_rs1_pairs",
                                  "many_items", "grouped", "nt96_fp32", "nt192"])
@pytest.mark.parametrize("fmt", ["bf16", "fp16"])
def test_pairs_on_off_bit_identical(name, fmt):
    """The same operands with and without CTA pairs give the same bits (measured on B200), so the engines' choice of
    pairs is invisible in their results."""
    c = CASES[name]
    p0, r0 = build(c, fmt, seed=5, pairs=False)
    p1, r1 = build(c, fmt, seed=5, pairs=True)
    p0.launch()
    p1.launch()
    torch.cuda.synchronize()
    d = (r0["out"].float() - r1["out"].float()).abs()
    print(json.dumps({"pairs_on_off": name, "fmt": fmt, "max_abs_diff": float(d.max()),
                      "n_diff": int((d > 0).sum())}), flush=True)
    assert torch.equal(r0["out"], r1["out"])


# ---------------------------------------------------------------------------------------------------- PDL chain
@pytest.mark.parametrize("fmt", ["bf16", "fp16"])
def test_pdl_chain_in_graph(fmt):
    """Two PDL plans captured in a graph as the wavefront decoder builds them: a torch kernel writes plan 1's input,
    plan 2 reads plan 1's output.  Replayed with new inputs; every replay is checked against the reference."""
    from masic_b200.convplan import ConvPlan, PackedConv
    dev = torch.device("cuda:0")
    dt = _dt(fmt)
    g = torch.Generator(device=dev).manual_seed(7)
    n, h, w = 1, 19, 34
    src = torch.empty(n, h, w, 128, device=dev)
    x = torch.zeros(n, h, w, 128, device=dev, dtype=dt)
    mid = torch.full((n, h, w, 384), SENTINEL, device=dev, dtype=dt)
    out = torch.full((n, h, w, 192), SENTINEL, device=dev, dtype=torch.float32)
    w1 = torch.randn(384, 128, 1, 1, device=dev, generator=g) / 128 ** 0.5
    b1 = torch.randn(384, device=dev, generator=g) * 0.1
    w2 = torch.randn(192, 384, 1, 1, device=dev, generator=g) / 384 ** 0.5
    b2 = torch.randn(192, device=dev, generator=g) * 0.1
    f16 = int(fmt == "fp16")
    pk1 = PackedConv(ksize=1, c_in=128, c_out=384, n_tile=192, weight=w1, bias=b1, f16=f16)
    pk2 = PackedConv(ksize=1, c_in=384, c_out=192, n_tile=192, weight=w2, bias=b2, f16=f16)
    acts = [R.ACT_RELU, R.ACT_LEAKY]
    p1 = ConvPlan(packed=pk1, x=x, out=mid, act=acts, pdl=True)
    p2 = ConvPlan(packed=pk2, x=mid, out=out, pdl=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(gr, stream=s):
            x.copy_(src)
            p1.launch()
            p2.launch()
    torch.cuda.current_stream().wait_stream(s)
    for rep in range(3):
        src.copy_(torch.randn(n, h, w, 128, device=dev, generator=g) * (1 + rep))
        out.fill_(SENTINEL)
        gr.replay()
        torch.cuda.synchronize()
        xin = src.to(dt)
        r1 = R.reference(ksize=1, x=xin, c_in=128, weight=w1, bias=b1, c_out=384, n_tile=192, out=mid, act=acts)
        q1, _ = R.ratio(mid, r1)
        r2 = R.reference(ksize=1, x=mid, c_in=384, weight=w2, bias=b2, c_out=192, n_tile=192,
                         out=torch.full_like(out, SENTINEL))
        q2, u2 = R.ratio(out, r2)
        print(json.dumps({"case": f"pdl_chain_replay{rep}", "fmt": fmt, "plan1": round(q1, 4), "plan2": round(q2, 4)}),
              flush=True)
        assert q1 <= 1.0 and q2 <= 1.0 and u2, (rep, q1, q2)


# ---------------------------------------------------------------------------------------------------- production plans
# Plans each builder creates; a change here means a plan was added or removed and must be audited (or skipped with a
# reason) on purpose.
EXPECTED_PLANS = {"hsic_engine": (41, 41), "wavefront_decoder": (10, 10), "hsic_trainer": (125, 125),
                  "cqe_engine": (42, 42), "lpips_engine": (5, 5), "udh_front_end": (8, 8)}


@pytest.fixture
def recorder(monkeypatch):
    """Records every ConvPlan built while the fixture is active, and the fp32 weights and bias every PackedConv was
    packed from (re-packs included)."""
    from masic_b200 import convplan
    plans = []
    pc_init, pc_repack, cp_init = convplan.PackedConv.__init__, convplan.PackedConv.repack, convplan.ConvPlan.__init__

    def rec_pc_init(self, *a, **kw):
        pc_init(self, *a, **kw)
        self._audit_w = kw["weight"].detach().float().clone()
        self._audit_b = None if kw.get("bias") is None else kw["bias"].detach().float().clone()

    def rec_pc_repack(self, weight, bias=None):
        pc_repack(self, weight, bias)
        self._audit_w = weight.detach().float().clone()
        if bias is not None:
            self._audit_b = bias.detach().float().clone()

    def rec_cp_init(self, *a, **kw):
        cp_init(self, *a, **kw)
        plans.append((self, kw))

    monkeypatch.setattr(convplan.PackedConv, "__init__", rec_pc_init)
    monkeypatch.setattr(convplan.PackedConv, "repack", rec_pc_repack)
    monkeypatch.setattr(convplan.ConvPlan, "__init__", rec_cp_init)
    return plans


def _overlaps(a, b):
    if a is None or b is None:
        return False
    sa, sb = a.untyped_storage(), b.untyped_storage()
    if sa.data_ptr() != sb.data_ptr():
        return False
    a0, a1 = a.data_ptr(), a.data_ptr() + a.numel() * a.element_size()
    b0, b1 = b.data_ptr(), b.data_ptr() + b.numel() * b.element_size()
    return a0 < b1 and b0 < a1


def audit(tag, plans):
    """Refill each recorded plan's inputs with fresh random values, launch it alone, compare with the reference."""
    from masic_b200 import _lib
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(11)
    torch.cuda.synchronize()
    n_done, worst = 0, 0.0
    for i, (plan, kw) in enumerate(plans):
        pk = plan.packed
        name = f"{tag}[{i}] {tuple(kw['x'].shape)}->{tuple(kw['out'].shape)} k{pk.ksize} kind{pk.kind} nt{pk.n_tile}"
        x, out = plan.x, plan.out
        act_out = getattr(plan, "act_out", None)
        ins = [x, *[r for r in plan.residuals if r is not None], plan.rowscale]
        if any(_overlaps(out, t) for t in ins) or any(_overlaps(act_out, t) for t in ins):
            print(json.dumps({"audit": name, "skipped": "output aliases an input"}), flush=True)
            continue
        with torch.no_grad():
            if not bool(pk._audit_w.any()):    # weights the builder leaves to the first training step's re-pack
                w = pk._audit_w
                pk.repack(torch.randn(w.shape, device=dev, generator=g) / (w[0].numel() ** 0.5))
            if pk.kind in (R.CONV_XFOLD4, R.CONV_XFOLD8):     # padded image rows: pad columns and unused channels 0
                x.zero_()
                wd = x.shape[2] - _lib.IMG_XPAD
                x[:, :, _lib.IMG_XOFF:_lib.IMG_XOFF + wd, :pk._audit_w.shape[1]] = torch.rand(
                    x.shape[0], x.shape[1], wd, pk._audit_w.shape[1], device=dev, generator=g).to(x.dtype)
            else:
                x.copy_(torch.randn(x.shape, device=dev, generator=g).to(x.dtype))
            for r in plan.residuals:
                if r is not None:
                    r.copy_(torch.randn(r.shape, device=dev, generator=g).to(r.dtype))
            if plan.rowscale is not None:
                plan.rowscale.copy_(torch.rand(plan.rowscale.shape, device=dev, generator=g) + 0.5)
            out.fill_(SENTINEL)
            if act_out is not None:
                act_out.fill_(SENTINEL)
        rkw = {k: v for k, v in kw.items() if k not in ("packed", "gdn_beta", "gdn_gamma")}
        rkw.update(kind=pk.kind, ksize=pk.ksize, c_in=pk.c_in, c_out=pk.c_out, n_tile=pk.n_tile,
                   c_out_pad=pk.c_out_pad, transposed=pk.transposed, weight=pk._audit_w, bias=pk._audit_b,
                   gdn=pk.gdn, beta_p=pk.beta, gamma_p=pk.gamma16, x=x, out=out, act_out=act_out)
        before = snapshot(rkw)
        plan.launch()
        torch.cuda.synchronize()
        r = R.reference(**{**rkw, **before})
        q, untouched = R.ratio(out, r)
        line = {"audit": name, "pairs": bool(kw.get("cta_pairs")), "pdl": bool(kw.get("pdl")),
                "max_err_over_bound": round(q, 4)}
        if act_out is not None:
            line["act_out_max_err_over_bound"] = round(R.ratio(act_out, r, act=True)[0], 4)
        print(json.dumps(line), flush=True)
        assert untouched and q <= 1.0, line
        assert line.get("act_out_max_err_over_bound", 0.0) <= 1.0, line
        worst = max(worst, q)
        n_done += 1
    print(json.dumps({"audit_summary": tag, "plans": len(plans), "audited": n_done, "worst": round(worst, 4)}),
          flush=True)
    return n_done


def _stereo(h, w, dev, seed=5):
    from oracle.hsic import synthetic_homography
    gg = torch.Generator().manual_seed(seed)
    x1, x2 = torch.rand(1, 3, h, w, generator=gg).to(dev), torch.rand(1, 3, h, w, generator=gg).to(dev)
    return x1, x2, synthetic_homography(1, seed=1).to(dev)


def _check_count(tag, plans, n_done):
    assert n_done > 0
    if tag in EXPECTED_PLANS:
        assert (len(plans), n_done) == EXPECTED_PLANS[tag], (tag, len(plans), n_done)


def test_audit_hsic_engine(recorder):
    from masic_b200.hsic import HSIC
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = HSIC().eval().to(dev)
    x1, x2, Hm = _stereo(128, 192, dev)
    with torch.no_grad():
        net(x1, x2, Hm)
    plans = list(recorder)
    _check_count("hsic_engine", plans, audit("hsic_engine", plans))


def test_audit_wavefront_decoder(recorder, tmp_path):
    from masic_b200.hsic import HSIC
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = HSIC().eval()
    with torch.no_grad():
        net.encoder1.g_a_conv4.weight.mul_(8.0)
        net.encoder2.g_a_conv4.weight.mul_(8.0)
    net = net.to(dev)
    net.update(force=True)
    x1, x2, Hm = _stereo(128, 192, dev)
    with torch.no_grad():
        net.compress(x1, x2, Hm, "pair0", str(tmp_path), y_order="wavefront")
        n0 = len(recorder)
        net.decompress(x1, x2, Hm, "pair0", str(tmp_path), device=dev)
    plans = [p for p in recorder[n0:] if p[1].get("pdl")]
    _check_count("wavefront_decoder", plans, audit("wavefront_decoder", plans))


def test_audit_hsic_trainer(recorder):
    from masic_b200.hsic import HSIC
    from masic_b200.trainer import HSICTrainer
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = HSIC().to(dev).train()
    HSICTrainer(net, 1, 64, 128, dev, lmbda=0.001)
    plans = list(recorder)
    _check_count("hsic_trainer", plans, audit("hsic_trainer", plans))


def test_audit_cqe_engine(recorder):
    from masic_b200.cqe import Independent_EN
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = Independent_EN().eval().to(dev)
    x1, x2, Hm = _stereo(64, 96, dev)
    with torch.no_grad():
        net(x1, x2, Hm)
    plans = list(recorder)
    _check_count("cqe_engine", plans, audit("cqe_engine", plans))


def test_audit_lpips_engine(recorder):
    from masic_b200.lpips import LPIPS
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = LPIPS(pretrained=False, pnet_rand=True, verbose=False).to(dev).eval()
    x1, x2, _ = _stereo(64, 96, dev)
    with torch.no_grad():
        net(x1, x2, normalize=True)
    plans = list(recorder)
    _check_count("lpips_engine", plans, audit("lpips_engine", plans))


def test_audit_cqe_trainer(recorder):
    from masic_b200.cqe import Independent_EN
    from masic_b200.cqe_trainer import CQETrainer
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = Independent_EN().to(dev).train()
    CQETrainer(net, 1, 64, 128, dev)
    plans = list(recorder)
    _check_count("cqe_trainer", plans, audit("cqe_trainer", plans))


def test_audit_udh_front_end(recorder):
    from masic_b200.udh import Net
    from oracle import udh as OU
    dev = torch.device("cuda:0")
    torch.manual_seed(1)
    net = Net().eval().to(dev)
    a, b, _ = OU.synthetic_patches(1, seed=2)
    with torch.no_grad():
        net(a.to(dev), b.to(dev))
    plans = list(recorder)
    _check_count("udh_front_end", plans, audit("udh_front_end", plans))
