"""The float64 conv reference (tests/conv_ref.py) and its per-element bound, checked without a GPU.

1. `conv_ref.reference` equals an independent loop coding in numpy to 1e-12: conv (3x3 stride 1, 5x5 stride 2,
   masked 5x5, the k=1 ConvTranspose2d), the stride-2 transposed conv in 4-phase and sub-pixel form, the XFOLD image
   input, a grouped table, planar output and rows wider than the image.
2. A simulated correct kernel output passes the bound: the float64 result plus accumulation noise of C_ACC * S,
   rounded to the output format.
3. Planted faults are rejected (max err / bound > 1) in each output format:
     relu        ReLU instead of LeakyReLU on one n-tile
     tap_slice   one 16-channel slice of one tap zeroed
     bias        the bias of one channel dropped
     rs_off±1    the rowscale read at rs_off - 1 / rs_off + 1
     tile_swap   one 16x8 tile's output taken from its neighbour
     res_coff    the residual read 8 channels off
   tools/conv_diag.run_case's old bar (max|got - ref| <= 1.2e-2 max|ref| for bf16 output, 1.5e-3 for fp16, 2e-3
   for fp32) accepts `relu` with bf16 output: ReLU instead of LeakyReLU moves a value by at most 0.01 of the largest
   output, under its 1.2e-2.  It rejects the other faults in this case, where each moves some element by more than
   the old bar; the new bound rejects every fault by a factor of 300 or more.  test_planted_fault asserts exactly
   this, so the statement stays true.
"""
from __future__ import annotations

import numpy as np
import pytest
import torch

import conv_ref as R
from conv_ref import (ACT_LEAKY, ACT_NONE, ACT_RELU, CONV, CONV_XFOLD4, CONV_XFOLD8, DECONV_S2, DECONV_S2_SUBPIX,
                      GDN_FWD, GDN_INV)


# ------------------------------------------------------------------ independent loop coding
def _conv_loops(x, w, stride, pad, mask=None, pad_x=None):
    """x (N, H, W, C), w (co, ci, k, k) correlation; zero padding `pad` rows and `pad_x` columns."""
    pad_x = pad if pad_x is None else pad_x
    n, h, wd, _ = x.shape
    co, ci, k, _ = w.shape
    ho, wo = (h + 2 * pad - k) // stride + 1, (wd + 2 * pad_x - k) // stride + 1
    out = np.zeros((n, ho, wo, co))
    for b in range(n):
        for oy in range(ho):
            for ox in range(wo):
                for ky in range(k):
                    for kx in range(k):
                        if mask is not None and not (mask >> (ky * k + kx)) & 1:
                            continue
                        iy, ix = oy * stride - pad + ky, ox * stride - pad_x + kx
                        if 0 <= iy < h and 0 <= ix < wd:
                            out[b, oy, ox] += w[:, :, ky, kx] @ x[b, iy, ix, :ci]
    return out


def _deconv_loops(x, w):
    """ConvTranspose2d(k=5, s=2, p=2, op=1): w (ci, co, 5, 5)."""
    n, h, wd, _ = x.shape
    out = np.zeros((n, 2 * h, 2 * wd, w.shape[1]))
    for b in range(n):
        for iy in range(h):
            for ix in range(wd):
                for ky in range(5):
                    for kx in range(5):
                        oy, ox = 2 * iy - 2 + ky, 2 * ix - 2 + kx
                        if 0 <= oy < 2 * h and 0 <= ox < 2 * wd:
                            out[b, oy, ox] += x[b, iy, ix] @ w[:, :, ky, kx]
    return out


def _act(v, a):
    return np.maximum(v, 0) if a == ACT_RELU else (np.where(v > 0, v, v * R.LEAKY_SLOPE) if a == ACT_LEAKY else v)


def _sq_np(y, dt):
    """The GDN norm operand: x^2 in fp32, rounded to bf16 to nearest even (bf16 plans) or half up (fp16 plans)."""
    y32 = y.astype(np.float32)
    bits = (y32 * y32).view(np.uint32).astype(np.uint64)
    if dt == torch.float16:
        bits = (bits + 0x8000) & 0xFFFF0000
    else:
        bits = (bits + 0x7FFF + ((bits >> 16) & 1)) & 0xFFFF0000
    return bits.astype(np.uint32).view(np.float32).astype(np.float64)


def _q(t, dt):
    return t.to(dt).double().numpy()


def _rnd(shape, dt, g, scale=1.0):
    return (torch.randn(*shape, generator=g) * scale).to(dt)


def _case(name, dt=torch.bfloat16, out_dt=None):
    """Tiny operands for one descriptor class.  Returns (ConvPlan-style kwargs, numpy expectation of `out`)."""
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    out_dt = out_dt or dt
    kw = {}
    if name in ("conv3", "conv5s2", "masked", "tconv1", "rowpix"):
        k, s, mask, tr = {"conv3": (3, 1, 0, False), "conv5s2": (5, 2, 0, False), "masked": (5, 1, R_MASK, False),
                          "tconv1": (1, 1, 0, True), "rowpix": (3, 1, 0, False)}[name]
        n, h, w, cin, cout, nt, cp, icoff = 2, 6, 4 if s == 2 else 5, 16, 24, 16, 40, 8
        x = _rnd((n, h, w + (3 if name == "rowpix" else 0), cp), dt, g)
        wt = torch.randn(*((cin, cout, k, k) if tr else (cout, cin, k, k)), generator=g)
        b = torch.randn(cout, generator=g)
        ho, wo = (h // s, w // s)
        out = torch.full((n, ho, wo, 48 + 8), 7.0).to(out_dt)
        acts = [ACT_LEAKY, ACT_RELU]
        rs = torch.rand(n, ho, wo, 3, generator=g) + 0.5
        res = _rnd((n, ho, wo, 48), dt, g) if s == 1 else None
        kw = dict(kind=CONV, ksize=k, stride=s, tap_mask=mask, x=x, in_coff=icoff, c_in=cin, weight=wt, transposed=tr,
                  bias=b, c_out=cout, n_tile=nt, out=out, out_coff=8, act=acts, rowscale=rs, rs_off=2,
                  residual0=res, res0_coff=8, w_in=w if name == "rowpix" else None)
        xin = _q(x, torch.float64)[..., icoff:icoff + cin]
        wq = _q(wt, dt)
        wc = np.flip(wq, (2, 3)).transpose(1, 0, 2, 3) if tr else wq
        pad_x = k // 2
        y = _conv_loops(xin, wc, s, k // 2, mask or None, pad_x)
        y = y[:, :, :wo]                                     # rowpix: taps past w read the buffer's own columns
        y = np.concatenate([y, np.zeros(y.shape[:3] + (32 - cout,))], -1) + np.concatenate([b.double().numpy(), np.zeros(8)])
        y = np.concatenate([_act(y[..., :16], acts[0]), _act(y[..., 16:], acts[1])], -1) * rs.double().numpy()[..., 2:3]
        if res is not None:
            y = y + _q(res, torch.float64)[..., 8:40]
        want = out.double().numpy().copy()
        want[..., 8:40] = y
        return kw, want
    if name in ("deconv", "subpix", "deconv_igdn"):
        n, h, w, cin = 1, 3, 4, 32
        cout = {"deconv": 24, "subpix": 3, "deconv_igdn": 128}[name]
        nt = {"deconv": 16, "subpix": 16, "deconv_igdn": 128}[name]
        x = _rnd((n, h, w, cin), dt, g)
        wt = torch.randn(cin, cout, 5, 5, generator=g) / 10
        b = torch.randn(cout, generator=g) * 0.1
        kind = DECONV_S2_SUBPIX if name == "subpix" else DECONV_S2
        y = _deconv_loops(_q(x, torch.float64), _q(wt, dt)) + b.double().numpy()
        extra = {}
        if name == "deconv_igdn":
            beta = torch.rand(cout, generator=g) + 0.5
            gam = (torch.rand(cout, cout, generator=g) * 0.01 + 0.1 * torch.eye(cout)).to(torch.bfloat16)
            extra = dict(gdn=GDN_INV, beta_p=beta, gamma_p=gam)
            norm = _sq_np(y, dt) @ gam.double().numpy().T + beta.double().numpy()
            y = y * np.sqrt(norm)
        if kind == DECONV_S2_SUBPIX:
            ys = np.zeros((n, h, w, 16))
            for py in range(2):
                for px in range(2):
                    ys[..., (py * 2 + px) * 3:(py * 2 + px) * 3 + 3] = y[:, py::2, px::2]
            ys[..., 12:] = 0.0
            y = ys
            out = torch.full((n, h, w, 16), 7.0).to(out_dt)
            want = y
        else:
            out = torch.full((n, 2 * h, 2 * w, (nt * -(-cout // nt))), 7.0).to(out_dt)
            want = np.concatenate([y, np.zeros(y.shape[:3] + (out.shape[3] - cout,))], -1)
            if name == "deconv":
                want = np.concatenate([_act(want[..., :16], ACT_LEAKY), _act(want[..., 16:], ACT_NONE)], -1)
        kw = dict(kind=kind, ksize=5, x=x, c_in=cin, weight=wt, transposed=True, bias=b, c_out=cout, n_tile=nt,
                  out=out, act=[ACT_LEAKY, ACT_NONE] if name == "deconv" else ACT_NONE, **extra)
        return kw, want
    if name in ("xfold4", "xfold8"):
        kind, cp = (CONV_XFOLD4, 16) if name == "xfold4" else (CONV_XFOLD8, 8)
        n, h, w, cout = 1, 6, 6, 16
        img = torch.rand(n, h, w, 3, generator=g)
        x = torch.zeros(n, h, w + R.IMG_XPAD, cp)
        x[:, :, R.IMG_XOFF:R.IMG_XOFF + w, :3] = img
        x = x.to(dt)
        wt = torch.randn(cout, 3, 5, 5, generator=g)
        b = torch.randn(cout, generator=g)
        beta = torch.rand(cout, generator=g) + 0.5
        gam = (torch.rand(cout, cout, generator=g) * 0.01 + 0.1 * torch.eye(cout)).to(torch.bfloat16)
        y = _conv_loops(_q(x, torch.float64)[:, :, R.IMG_XOFF:R.IMG_XOFF + w, :3], _q(wt, dt), 2, 2) + b.double().numpy()
        y = y / np.sqrt(_sq_np(y, dt) @ gam.double().numpy().T + beta.double().numpy())
        out = torch.full((n, h // 2, w // 2, cout), 7.0).to(out_dt)
        kw = dict(kind=kind, ksize=5, stride=2, x=x, c_in=64, weight=wt, bias=b, c_out=cout, n_tile=cout, out=out,
                  gdn=GDN_FWD, beta_p=beta, gamma_p=gam)
        return kw, y
    if name == "grouped":
        n, h, w, K = 2, 3, 5, 16
        x = _rnd((n, h, w, 3 * K), dt, g)
        wt = torch.randn(64, K, 1, 1, generator=g)
        b = torch.randn(64, generator=g)
        out = torch.full((3 * n, h, w, 40), 7.0).to(out_dt)
        tin, toc, toi = [0, K, 2 * K, 2 * K], [0, 8, 0, 16], [0, n, 2 * n, 2 * n]
        acts = [ACT_RELU, ACT_NONE, ACT_LEAKY, ACT_LEAKY]
        want = out.double().numpy().copy()
        for t in range(4):
            xs = _q(x, torch.float64)[..., tin[t]:tin[t] + K]
            y = _conv_loops(xs, _q(wt, dt)[16 * t:16 * t + 16], 1, 0) + b.double().numpy()[16 * t:16 * t + 16]
            want[toi[t]:toi[t] + n, ..., 8 + toc[t]:8 + toc[t] + 16] = _act(y, acts[t])
        kw = dict(ksize=1, x=x, c_in=K, weight=wt, bias=b, c_out=64, n_tile=16, out=out, out_coff=8, act=acts,
                  nt_in_coff=tin, nt_out_coff=toc, nt_out_img=toi)
        return kw, want
    if name == "planar":
        n, h, w = 2, 4, 5
        x = _rnd((n, h, w, 64), dt, g)
        wt = torch.randn(48, 64, 3, 3, generator=g)
        b = torch.randn(48, generator=g)
        fp32 = out_dt == torch.float32
        bc = 16 if fp32 else 48
        nblk = 48 // bc
        out = torch.full((n * nblk, h, w, 8), 7.0).to(out_dt)
        y = _conv_loops(_q(x, torch.float64), _q(wt, dt), 1, 1) + b.double().numpy()
        want = out.double().numpy().copy()
        for bb in range(n):
            for j in range(nblk):
                want[bb * nblk + j] = y[bb, ..., j * bc:j * bc + 8]          # channels past out_cpitch are clipped
        kw = dict(ksize=3, x=x, c_in=64, weight=wt, bias=b, c_out=48, n_tile=48, out=out, out_blk_images=True)
        return kw, want
    raise KeyError(name)


R_MASK = sum(1 << (ky * 5 + kx) for ky in range(5) for kx in range(5) if ky < 2 or (ky == 2 and kx < 2))
NAMES = ["conv3", "conv5s2", "masked", "tconv1", "rowpix", "deconv", "subpix", "deconv_igdn", "xfold4", "xfold8",
         "grouped", "planar"]


@pytest.mark.parametrize("out_fp32", [False, True])
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("name", NAMES)
def test_reference_matches_loops(name, dt, out_fp32):
    kw, want = _case(name, dt, torch.float32 if out_fp32 else dt)
    r = R.reference(**kw)
    got = r.ref.numpy()
    if name == "subpix":
        got = got[..., :16]
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    # the elements the plan leaves alone are exactly those that kept the sentinel in the loop coding
    assert np.array_equal(~r.written.numpy(), (want == 7.0)) or name in ("subpix", "xfold4", "xfold8", "deconv_igdn")


def _simulated(r: R.Ref, g, frac=0.5, c_acc=None):
    """A correct kernel's output: the exact value plus accumulation noise inside the bound, rounded to the format."""
    c_acc = R.C_ACC if c_acc is None else c_acc
    noise = (torch.rand(r.ref.shape, generator=g, dtype=torch.float64) * 2 - 1) * frac * c_acc * r.mag
    v = R.round_to(r.ref + noise, r.out_fmt)
    return torch.where(r.written, v, r.ref)


@pytest.mark.parametrize("out_fp32", [False, True])
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("name", NAMES)
def test_simulated_kernel_passes(name, dt, out_fp32):
    kw, _ = _case(name, dt, torch.float32 if out_fp32 else dt)
    r = R.reference(**kw)
    q, untouched = R.ratio(_simulated(r, torch.Generator().manual_seed(1)), r)
    assert untouched and q <= 1.0, q


def test_fp16_saturates():
    x = torch.full((1, 16, 8, 16), 8.0).to(torch.float16)
    w = torch.full((16, 16, 1, 1), 1000.0)
    out = torch.zeros(1, 16, 8, 16, dtype=torch.float16)
    r = R.reference(ksize=1, x=x, c_in=16, weight=w, c_out=16, n_tile=16, out=out)
    assert float(r.ref.max()) == R.F16_MAX
    got = torch.full_like(r.ref, R.F16_MAX)
    assert R.ratio(got, r)[0] <= 1.0
    assert R.ratio(torch.full_like(r.ref, float("inf")), r)[0] == float("inf")


# ------------------------------------------------------------------ planted faults
def _fault_case(fmt):
    """3x3 conv, three 32-wide n-tiles (ReLU / LeakyReLU / none), rowscale (stride 3, rs_off 1), one residual at a
    channel offset: every epilogue input the faults can disturb.  Outputs ~N(0, 1), like the gmm_l0 case."""
    g = torch.Generator().manual_seed(3)
    dt = torch.float16 if fmt == "fp16" else torch.bfloat16
    out_dt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[fmt]
    n, h, w, cin, cout = 1, 20, 20, 64, 96
    x = _rnd((n, h, w, cin), dt, g)
    wt = torch.randn(cout, cin, 3, 3, generator=g) / (9 * cin) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    rs = torch.rand(n, h, w, 3, generator=g) + 0.5
    res = _rnd((n, h, w, cout + 16), dt, g)
    out = torch.full((n, h, w, cout), 7.0).to(out_dt)
    return dict(ksize=3, x=x, c_in=cin, weight=wt, bias=b, c_out=cout, n_tile=32, out=out,
                act=[ACT_RELU, ACT_LEAKY, ACT_NONE], rowscale=rs, rs_off=1, residual0=res, res0_coff=8)


def _faulty(kw, fault):
    kw = dict(kw)
    if fault == "relu":
        kw["act"] = [ACT_RELU, ACT_RELU, ACT_NONE]
    elif fault == "tap_slice":
        wt = kw["weight"].clone()
        wt[:, 16:32, 1, 2] = 0.0
        kw["weight"] = wt
    elif fault == "bias":
        b = kw["bias"].clone()
        b[40] = 0.0
        kw["bias"] = b
    elif fault in ("rs_off-1", "rs_off+1"):
        kw["rs_off"] = kw["rs_off"] + (1 if fault.endswith("+1") else -1)
    elif fault == "res_coff":
        kw["res0_coff"] = kw["res0_coff"] + 8
    r = R.reference(**kw)
    got = R.round_to(r.ref, r.out_fmt)
    if fault == "tile_swap":                          # tile (ty 0, tx 0) holds tile (ty 0, tx 1)'s values
        got[:, 0:16, 0:8] = got[:, 0:16, 8:16]
    return got


FAULTS = ["relu", "tap_slice", "bias", "rs_off-1", "rs_off+1", "tile_swap", "res_coff"]
OLD_BAR_ACCEPTS = {("relu", "bf16")}


@pytest.mark.parametrize("fmt", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("fault", FAULTS)
def test_planted_fault(fault, fmt):
    kw = _fault_case(fmt)
    r = R.reference(**kw)
    assert R.ratio(R.round_to(r.ref, r.out_fmt), r)[0] <= 1.0          # the fault-free output passes
    got = _faulty(kw, fault)
    q, _ = R.ratio(got, r)
    assert q > 1.0, (fault, fmt, q)
    assert R.old_bar_accepts(got, r) == ((fault, fmt) in OLD_BAR_ACCEPTS), (fault, fmt)
