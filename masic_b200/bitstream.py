"""HSIC.compress / HSIC.decompress on the sm_100a kernels (reference: coremasic/mywork/MASIC.py:855-1158, :1161-1408).

What the reference does, and what is kept:
  * side information: `EntropyBottleneck.compress` of z1, z2 through the reference's rANS extension, behind the
    same file header (`<name>.npz`: uint16 H, W | uint16 len(z1), minmax1 | M/8-byte non-zero-channel bitmap | z1 |
    uint16 len(z2), minmax2 | bitmap | z2 — MASIC.py:922-952).  Byte-identical given identical z symbols.
  * y1, y2: one range-coded symbol per (row, column, non-zero channel) in raster order, each under its own
    integer CDF built from the K=5 Gaussian-mixture parameters by the rule of MASIC.py:1006-1043.  The encoder
    knows y_hat, so ALL parameters come from one forward pass of the engine and ALL coding intervals from one
    kernel (`masic_gmm_symbol_cdfs`) — the reference recomputes the context model and the parameter nets per
    pixel in Python.  The decoder is autoregressive (the mask-A context conv needs the already-decoded
    neighbourhood) and walks the pixels in order, evaluating the SAME conv kernels on a 5x5 crop / a single
    pixel so that it reproduces the encoder's parameters bit for bit.
  * symbol ORDER inside `<name>.bin`: the reference codes raster order, which forces a decoder to finish row h-1
    before it can start row h.  The mask-A 5x5 context of position (h, w) only reaches columns w-2..w+2 of the two
    rows above and w-2, w-1 of its own row, so every position of the anti-diagonal wave t = w + 3h depends on
    earlier waves only (SURVEY 8(f)#3).  By default both sides therefore code the positions in WAVE order
    (t ascending, h ascending inside a wave; first payload byte = 1): the decoder evaluates the context conv, the
    parameter nets and the CDF rows of a whole wave (up to ceil(W/48)+1 positions) in one batch and range-decodes
    their symbols in one host call - (W/16 + 3(H/16-1)) steps instead of H*W/256.  `y_order="raster"` (payload
    byte 0) keeps the reference's order and the per-position decoder.  The CDFs, hence the code length, are the
    same either way.
  * format 2 (the default, one range-coded stream per (view, non-zero channel)) is coded for a whole batch of pairs of
    one size at once: `compress_batch` runs one batch-B forward pass and one device encoder launch for every stream of
    every pair; `decompress_batch` walks the shared wave schedule once, each wave's launches covering all pairs.  Each
    pair keeps its own reference-layout header and payload; `compress` / `decompress` are the B = 1 case.
  * the range coder itself: the reference calls the PyPI package `range_coder`, which it neither vendors nor
    pins and which is not installable here; `masic_range_encode` / `masic_range_decode_rows` (csrc/cdf.cu) are a
    plain 32-bit range coder with the same interface.  `<name>.bin` therefore has this library's byte format.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from ._lib import MasicError, check
from .convplan import ACT_LEAKY, ACT_NONE, ACT_RELU, MASK_A_5x5, ConvPlan
from .engine import ACT, SCALE_BOUND, HSICEngine
from .ops import _f32c
from .padding import Padding, padding_for, run_engine


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _nonzero_channels(y_hat_nchw: torch.Tensor):
    """MASIC.py:925-940: bitmap of channels with any non-zero symbol, and minmax = max(|y_hat|, 1)."""
    a = y_hat_nchw.abs()
    flag = (a.sum(dim=(0, 2, 3)) > 0).to(torch.uint8).cpu().numpy().astype(np.int64)
    minmax = int(max(float(a.max()), 1.0))
    return flag, minmax


def _pack_flags(flag: np.ndarray) -> bytes:
    # np.packbits(np.reshape(flag, [8, M // 8])) flattens first: identical to packing the flat array (MASIC.py:932)
    return np.packbits(np.reshape(flag, [8, flag.shape[0] // 8])).astype(np.uint8).tobytes()


class _PixelModel:
    """GMM parameters of ONE latent position through the engine's own conv kernels: the mask-A context conv on a
    5x5 crop of the decoded latents, then the three 1x1 parameter branches on a 1-pixel image."""

    def __init__(self, eng: HSICEngine, tag: str):
        M, K, dev = eng.M, eng.K, eng.dev
        self.eng, self.tag, self.M, self.K = eng, tag, M, K
        self.right = tag == "R"
        cin = 5 * M if self.right else 4 * M
        MK = M * K
        bf, f32 = ACT, torch.float32
        z = lambda *s, dtype=bf: torch.zeros(*s, dtype=dtype, device=dev)   # noqa: E731
        self.crop = z(1, 5, 5, M)
        self.ctx_out = z(1, 5, 5, cin)
        self.rs = z(1, 5, 5, 3, dtype=f32) if self.right else None
        self.px_in = z(1, 1, 1, cin)
        self.l0, self.l1, self.l1w = z(1, 1, 1, 18 * M), z(1, 1, 1, 8 * M), z(1, 1, 1, MK)
        self.sig, self.mu, self.wl = z(1, 1, 1, MK, dtype=f32), z(1, 1, 1, MK, dtype=f32), z(1, 1, 1, MK, dtype=f32)
        pk = eng.packs
        # exactly the epilogue configuration of HSICEngine._build / _gmm_net
        self.plans = [
            ConvPlan(packed=pk[f"{tag}.context"], stride=1, tap_mask=MASK_A_5x5, x=self.crop, out=self.ctx_out,
                     out_coff=2 * M, rowscale=self.rs, rs_off=1)]
        self.tail = [
            ConvPlan(packed=pk[f"{tag}.gmm.l0"], x=self.px_in, out=self.l0, act=[ACT_RELU] * 6 + [ACT_LEAKY] * 12),
            ConvPlan(packed=pk[f"{tag}.gmm.sigma.l1"], x=self.l0, out=self.l1, in_coff=0, out_coff=0, act=ACT_RELU),
            ConvPlan(packed=pk[f"{tag}.gmm.means.l1"], x=self.l0, out=self.l1, in_coff=6 * M, out_coff=4 * M, act=ACT_LEAKY),
            ConvPlan(packed=pk[f"{tag}.gmm.weights.l1"], x=self.l0, out=self.l1w, in_coff=12 * M, act=ACT_LEAKY),
            ConvPlan(packed=pk[f"{tag}.gmm.sigma.l2"], x=self.l1, out=self.sig, in_coff=0, act=ACT_RELU),
            ConvPlan(packed=pk[f"{tag}.gmm.means.l2"], x=self.l1, out=self.mu, in_coff=4 * M),
            ConvPlan(packed=pk[f"{tag}.gmm.weights.l2"], x=self.l1w, out=self.wl),
        ]

    def params_at(self, ypad: torch.Tensor, gmm_in: torch.Tensor, h: int, w: int):
        M = self.M
        self.crop.copy_(ypad[:, h:h + 5, w:w + 5, :])
        if self.right:
            self.rs.copy_(self.eng.mask_weights[:, h:h + 1, w:w + 1, :].expand(1, 5, 5, 3))
        self.plans[0].launch()
        self.px_in[..., :2 * M].copy_(gmm_in[:, h:h + 1, w:w + 1, :2 * M])
        self.px_in[..., 2 * M:4 * M].copy_(self.ctx_out[:, 2:3, 2:3, 2 * M:4 * M])
        if self.right:
            self.px_in[..., 4 * M:].copy_(gmm_in[:, h:h + 1, w:w + 1, 4 * M:])
        for p in self.tail:
            p.launch()
        return self.sig, self.mu, self.wl


ORDER_RASTER, ORDER_WAVE, ORDER_WAVE_STREAMS = 0, 1, 2
_ORDERS = {"raster": ORDER_RASTER, "wavefront": ORDER_WAVE, "wavefront_streams": ORDER_WAVE_STREAMS}


def wave_schedule(h16: int, w16: int):
    """Positions (raster index h*w16 + w) grouped by wave t = w + 3h, h ascending inside a wave."""
    waves = []
    for t in range(w16 + 3 * (h16 - 1)):
        hs = np.arange(max(0, -(-(t - w16 + 1) // 3)), min(h16 - 1, t // 3) + 1, dtype=np.int64)
        ws = t - 3 * hs
        keep = (ws >= 0) & (ws < w16)
        if keep.any():
            waves.append((hs[keep], ws[keep]))
    return waves


def wave_permutation(h16: int, w16: int) -> np.ndarray:
    return np.concatenate([hs * w16 + ws for hs, ws in wave_schedule(h16, w16)])


class _WaveModel:
    """GMM parameters of all positions of one wave through the engine's own conv kernels: the mask-A context conv on
    a batch of 5x5 crops of the decoded latents, then the 1x1 parameter branches on a (1, 1, n, C) image.  Row results
    of an MMA do not depend on the other rows, so every position gets bit for bit what the encoder's full-image
    launches produced."""

    def __init__(self, eng: HSICEngine, tag: str, n_max: int):
        M, K, dev = eng.M, eng.K, eng.dev
        self.eng, self.tag, self.M, self.K, self.n_max = eng, tag, M, K, n_max
        self.right = tag == "R"
        cin = 5 * M if self.right else 4 * M
        self.cin = cin
        MK = M * K
        bf, f32 = ACT, torch.float32
        z = lambda *s, dtype=bf: torch.zeros(*s, dtype=dtype, device=dev)   # noqa: E731
        self.crop = z(n_max, 5, 5, M)
        self.ctx_out = z(n_max, 5, 5, cin)
        self.rs = z(n_max, 5, 5, 3, dtype=f32) if self.right else None
        self.px_in = z(1, 1, n_max, cin)
        # the parameter nets exactly as HSICEngine._gmm_net launches them: layer 0 of the three branches as one wide
        # GEMM, layer 1 as one grouped launch, layer 2 as sigma|means grouped + weights (4 launches instead of 7)
        self.l0, self.l1 = z(1, 1, n_max, 18 * M), z(1, 1, n_max, 13 * M)
        smw = z(3, 1, n_max, MK, dtype=f32)
        self.sig, self.mu, self.wl = smw[0:1], smw[1:2], smw[2:3]
        pk = eng.packs
        nt = lambda c: c // 192   # noqa: E731
        tiles = list(range(0, MK, 192))
        self.ctx_plan = ConvPlan(packed=pk[f"{tag}.context"], stride=1, tap_mask=MASK_A_5x5, x=self.crop,
                                 out=self.ctx_out, out_coff=2 * M, rowscale=self.rs, rs_off=1, pdl=True)
        self.tail = [
            ConvPlan(packed=pk[f"{tag}.gmm.l0"], x=self.px_in, out=self.l0, act=[ACT_RELU] * 6 + [ACT_LEAKY] * 12, pdl=True),
            ConvPlan(packed=pk[f"{tag}.gmm.l1(3 branches)"], x=self.l0, out=self.l1,
                     act=[ACT_RELU] * nt(4 * M) + [ACT_LEAKY] * nt(9 * M),
                     nt_in_coff=[0] * nt(4 * M) + [6 * M] * nt(4 * M) + [12 * M] * nt(5 * M), pdl=True),
            ConvPlan(packed=pk[f"{tag}.gmm.l2(sigma|means)"], x=self.l1, out=smw, act=[ACT_RELU] * nt(MK) + [ACT_NONE] * nt(MK),
                     nt_in_coff=[0] * nt(MK) + [4 * M] * nt(MK), nt_out_coff=tiles + tiles,
                     nt_out_img=[0] * nt(MK) + [1] * nt(MK), pdl=True),
            ConvPlan(packed=pk[f"{tag}.gmm.weights.l2"], x=self.l1, out=self.wl, in_coff=8 * M, pdl=True),
        ]

    def params_at(self, ypad_flat: torch.Tensor, gmm_flat: torch.Tensor, crop_idx: torch.Tensor, pos: torch.Tensor):
        """ypad_flat ((h16+4)*(w16+4), M) bf16, gmm_flat (h16*w16, cin) bf16, crop_idx (n*25,) / pos (n,) int64."""
        M, n = self.M, pos.numel()
        self.crop.view(-1, M)[:n * 25].copy_(ypad_flat.index_select(0, crop_idx))
        if self.right:
            mw = self.eng.mask_weights.view(-1, 3).index_select(0, pos)
            self.rs[:n].copy_(mw.view(n, 1, 1, 3).expand(n, 5, 5, 3))
        self.ctx_plan.launch()
        g = gmm_flat.index_select(0, pos)
        px = self.px_in.view(self.n_max, self.cin)
        px[:n, :2 * M].copy_(g[:, :2 * M])
        px[:n, 2 * M:4 * M].copy_(self.ctx_out[:n, 2, 2, 2 * M:4 * M])
        if self.right:
            px[:n, 4 * M:].copy_(g[:, 4 * M:])
        for p in self.tail:
            p.launch()
        return self.sig, self.mu, self.wl


def _symbol_intervals(eng: HSICEngine, tag: str, y_hat_nchw: torch.Tensor, ch: torch.Tensor, minmax: int) -> np.ndarray:
    """(n_pos * n_ch, 3) int32 coding intervals of every listed latent element, raster order, channel-minor."""
    lib = eng.lib
    M, K = eng.M, eng.K
    y_nhwc = y_hat_nchw.permute(0, 2, 3, 1).contiguous()
    n_pos = y_nhwc.shape[1] * y_nhwc.shape[2]
    out = torch.empty(n_pos * ch.numel(), 3, dtype=torch.int32, device=eng.dev)
    check(lib.masic_gmm_symbol_cdfs(eng.buf[f"{tag}.sigma"].data_ptr(), eng.buf[f"{tag}.mu"].data_ptr(),
                                    eng.buf[f"{tag}.wlogit"].data_ptr(), 1, M, K, n_pos, ch.data_ptr(), ch.numel(),
                                    minmax, SCALE_BOUND, y_nhwc.data_ptr(), None, out.data_ptr(), _stream()),
          "masic_gmm_symbol_cdfs")
    return out.cpu().numpy()


def _header_bytes(H: int, W: int, z_strings, minmaxs, flags) -> bytes:
    """`<name>.npz` (MASIC.py:922-952): uint16 H, W | per view: uint16 len(z), minmax | bitmap | z."""
    parts = [np.array([H, W], dtype=np.uint16).tobytes()]
    for zs, mm, fl in zip(z_strings, minmaxs, flags):
        if len(zs) > 65535:
            raise MasicError("z bitstream exceeds the uint16 length field of the reference header (MASIC.py:945)")
        parts += [np.array([len(zs), mm], dtype=np.uint16).tobytes(), _pack_flags(fl), zs]
    return b"".join(parts)


def _z_strings(model, eng: HSICEngine):
    """Side information of every pair through the reference rANS (entropy_models.py:420-423): [view][pair] bytes."""
    return [eb.compress(eng.buf[f"{tag}.z"].permute(0, 3, 1, 2).contiguous())
            for tag, eb in (("L", model.entropy_bottleneck1), ("R", model.entropy_bottleneck2))]


def _stream_table(flags: np.ndarray, minmax: np.ndarray) -> np.ndarray:
    """(3, S) int32 pair | channel | minmax of the streams of one view, pair-major (flags (B, M), minmax (B,))."""
    pair, ch = np.nonzero(flags)
    return np.ascontiguousarray(np.stack([pair, ch, minmax[pair]]).astype(np.int32))


def _stream_intervals(eng: HSICEngine, tag: str, y_hat_nchw: torch.Tensor, table: torch.Tensor, max_minmax: int,
                      out: torch.Tensor) -> None:
    """Coding intervals of every stream of one view into out (n_pos, S, 3) int32, raster order."""
    M, K = eng.M, eng.K
    n_pos = out.shape[0]
    y_nhwc = y_hat_nchw.permute(0, 2, 3, 1).contiguous()
    check(eng.lib.masic_gmm_symbol_cdfs_pairs(
        eng.buf[f"{tag}.sigma"].data_ptr(), eng.buf[f"{tag}.mu"].data_ptr(), eng.buf[f"{tag}.wlogit"].data_ptr(), 1, M, K,
        n_pos, n_pos, table[0].data_ptr(), table[1].data_ptr(), table[2].data_ptr(), table.shape[1], max_minmax,
        SCALE_BOUND, y_nhwc.data_ptr(), None, 0, out.data_ptr(), _stream()), "masic_gmm_symbol_cdfs_pairs")


def _encode_pairs(model, eng: HSICEngine, pad: Padding, y_clock: Optional[list] = None):
    """Format-2 header and payload of every pair of the engine's last forward pass.  The intervals of all streams of
    both views are computed, put in wave order and range-coded on the device; only the packed payload bytes, the
    stream offsets and the flags are read back.  y_clock, if given, receives time.time() where the y coding starts.
    y_bits_ideal is summed per stream on the device, then over the pair's streams (float64).  The header holds the
    pair's own size `pad.h`, `pad.w`; the latents are those of the padded frame the engine ran on."""
    lib, dev = eng.lib, eng.dev
    B, H, W, M = eng.B, eng.H, eng.W, eng.M
    n_pos = (H // 16) * (W // 16)
    z_strings = _z_strings(model, eng)
    # non-zero-channel bitmaps and minmax = max(|y_hat|, 1) of every pair and view (MASIC.py:925-940), one read-back
    a = [eng.out[k].abs() for k in ("y1_hat", "y2_hat")]
    small = torch.cat([torch.stack([(t.sum(dim=(2, 3)) > 0).float() for t in a]).flatten(),
                       torch.stack([t.amax(dim=(1, 2, 3)).clamp_min(1.0) for t in a]).flatten()]).cpu().numpy()
    flags = small[:2 * B * M].reshape(2, B, M).astype(np.int64)
    minmax = small[2 * B * M:].reshape(2, B).astype(np.int64)
    headers = [_header_bytes(pad.h, pad.w, [z_strings[0][b], z_strings[1][b]], minmax[:, b], flags[:, b])
               for b in range(B)]
    tables = [_stream_table(flags[v], minmax[v]) for v in range(2)]
    S = [t.shape[1] for t in tables]
    n_streams = S[0] + S[1]
    iv = torch.empty(n_pos * n_streams * 3, dtype=torch.int32, device=dev)
    slot_cap = 3 * n_pos + 16
    slots = torch.empty(n_streams * slot_cap, dtype=torch.uint8, device=dev)
    # the packed payload goes over the intervals: 12 * n_pos bytes per stream exceed slot_cap, and the encoder has read
    # every interval before the packing launch (same stream) writes there
    packed = iv.view(torch.uint8)
    lens = torch.zeros(n_streams, dtype=torch.int64, device=dev)
    offs = torch.zeros(n_streams + 1, dtype=torch.int64, device=dev)
    bits = torch.zeros(n_streams, dtype=torch.float64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    if y_clock is not None:
        y_clock.append(time.time())
    if n_streams:
        perm = torch.from_numpy(wave_permutation(H // 16, W // 16)).to(dev)
        base, stride, o = [], [], 0
        for v, tag in enumerate(("L", "R")):
            if not S[v]:
                continue
            view = iv[o * 3:(o + n_pos * S[v]) * 3].view(n_pos, S[v], 3)
            _stream_intervals(eng, tag, eng.out[("y1_hat", "y2_hat")[v]], torch.from_numpy(tables[v]).to(dev),
                              int(tables[v][2].max()), view)
            view.copy_(view.index_select(0, perm))          # positions in wave order, streams stay minor
            k = S[0] if v else 0
            for p0 in range(0, n_pos, 2048):               # float64 in slices: a whole view would be 16 B per interval
                f = view[p0:p0 + 2048, :, 1:].double()
                bits[k:k + S[v]] -= torch.log2(f[..., 0] / f[..., 1]).sum(0)
            base.append(o + np.arange(S[v]))
            stride.append(np.full(S[v], S[v]))
            o += n_pos * S[v]
        base_d = torch.from_numpy(np.concatenate(base).astype(np.int64)).to(dev)
        stride_d = torch.from_numpy(np.concatenate(stride).astype(np.int64)).to(dev)
        check(lib.masic_range_encode_streams(iv.data_ptr(), base_d.data_ptr(), stride_d.data_ptr(), n_pos, n_streams,
                                             slots.data_ptr(), slot_cap, lens.data_ptr(), err.data_ptr(), _stream()),
              "masic_range_encode_streams")
        check(lib.masic_pack_streams(slots.data_ptr(), slot_cap, lens.data_ptr(), n_streams, offs.data_ptr(),
                                     packed.data_ptr(), _stream()), "masic_pack_streams")
    meta = torch.cat([err.double(), offs.double(), bits]).cpu().numpy()
    if meta[0]:
        raise MasicError("y payload: an invalid coding interval (empty, outside the total, or total > 2^22)")
    offs_h = meta[1:n_streams + 2].astype(np.int64)
    bits_h = meta[n_streams + 2:]
    data = packed[:int(offs_h[-1])].cpu().numpy().tobytes()
    # stream ranges of every (view, pair): the tables are pair-major
    first = [np.searchsorted(t[0], np.arange(B + 1)) + (S[0] if v else 0) for v, t in enumerate(tables)]
    items = []
    for b in range(B):
        parts, n_sym, ideal = [bytes([ORDER_WAVE_STREAMS])], 0, 0.0
        for v in range(2):
            s0, s1 = int(first[v][b]), int(first[v][b + 1])
            parts += [np.array([s1 - s0], dtype=np.uint32).tobytes()]
            if s1 > s0:
                parts += [np.diff(offs_h[s0:s1 + 1]).astype(np.uint32).tobytes(), data[offs_h[s0]:offs_h[s1]]]
            n_sym += n_pos * (s1 - s0)
            ideal += float(bits_h[s0:s1].sum())
        payload = b"".join(parts)
        items.append({"header": headers[b], "payload": payload,
                      "bpp_real": (len(headers[b]) + len(payload)) * 8 / (2 * pad.h * pad.w),
                      "n_symbols": n_sym, "y_bits_ideal": ideal})
    return items


def _check_inputs(model, what: str, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor) -> None:
    if model.training:
        raise MasicError(f"{what}: eval mode only")
    if not (x1.is_cuda and x2.is_cuda and h_matrix.is_cuda):
        raise MasicError(f"{what} needs CUDA tensors: masic_b200 has no CPU fallback")
    if x1.dim() != 4 or x2.shape != x1.shape:
        raise ValueError(f"{what}: x1 and x2 must be (B, 3, H, W) tensors of one shape")
    if h_matrix.numel() != 9 * x1.shape[0]:
        raise ValueError(f"{what}: h_matrix must hold one 3x3 homography per pair, got {tuple(h_matrix.shape)}")


def compress_batch(model, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor):
    """Code B pairs of one size at once: one batch-B forward pass, one device encoder launch for every stream.  Returns
    one dict per pair: `header` / `payload` are the bytes of its `<name>.npz` / `<name>.bin` (format 2), identical to
    what `compress` writes for that pair alone; `bpp_real`, `n_symbols`, `y_bits_ideal` as in `compress`."""
    _check_inputs(model, "HSIC.compress_batch", x1, x2, h_matrix)
    B, _, H, W = x1.shape
    pad = padding_for(H, W)
    pad.check_header()
    eng: HSICEngine = model.engine_for(B, pad.hp, pad.wp, x1.device)
    with torch.cuda.device(eng.dev):
        run_engine(eng, pad, x1, x2, h_matrix)
        return _encode_pairs(model, eng, pad)


def compress(model, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor, output_name, output_path: str = "",
             device=None, y_order: str = "wavefront_streams") -> Dict:
    """HSIC.compress (MASIC.py:855-1158).  Batch 1, like the reference's file format.  `enctime` covers the y coding
    and the writing of the payload; with the default order `y_bits_ideal` is summed per stream first (see
    `_encode_pairs`), so its last bits can differ from one sum over all intervals."""
    if model.training:
        raise MasicError("HSIC.compress: eval mode only")
    if x1.shape[0] != 1:
        raise ValueError("HSIC.compress writes one stereo pair per file (MASIC.py:922: a single H, W header)")
    if y_order not in _ORDERS:
        raise ValueError(f'y_order must be one of {sorted(_ORDERS)}, got {y_order!r}')
    order = _ORDERS[y_order]
    lib = _lib.load()
    pad = padding_for(*x1.shape[2:])
    pad.check_header()
    H, W = pad.hp, pad.wp                   # the coded latents are those of the padded frame
    eng: HSICEngine = model.engine_for(1, H, W, x1.device)
    out = run_engine(eng, pad, x1, x2, h_matrix)
    output1 = os.path.join(output_path, str(output_name) + ".npz")
    output2 = os.path.join(output_path, str(output_name) + ".bin")
    if order == ORDER_WAVE_STREAMS:
        # one range-coded stream per (view, non-zero channel): | 2 | per view: u32 n_ch, u32 len[n_ch], streams |
        clock = []
        item = _encode_pairs(model, eng, pad, clock)[0]
        with open(output1, "wb") as f:
            f.write(item["header"])
        with open(output2, "wb") as f:
            f.write(item["payload"])
        start, end = clock[0], time.time()
        n_symbols, ideal_bits = item["n_symbols"], item["y_bits_ideal"]
    else:
        z_strings = _z_strings(model, eng)
        y_hats = {"L": out["y1_hat"], "R": out["y2_hat"]}
        flags, minmaxs = {}, {}
        for tag in ("L", "R"):
            flags[tag], minmaxs[tag] = _nonzero_channels(y_hats[tag])
        with open(output1, "wb") as f:
            f.write(_header_bytes(pad.h, pad.w, [zs[0] for zs in z_strings], [minmaxs["L"], minmaxs["R"]],
                                  [flags["L"], flags["R"]]))
        # ---- y1, y2: all coding intervals in one kernel each, one range-coded stream
        start = time.time()
        perm = wave_permutation(H // 16, W // 16) if order != ORDER_RASTER else None
        ivs = []
        for tag in ("L", "R"):
            ch = torch.from_numpy(np.flatnonzero(flags[tag]).astype(np.int32)).to(eng.dev)
            if ch.numel():
                a = _symbol_intervals(eng, tag, y_hats[tag], ch, minmaxs[tag])
                if perm is not None:          # positions in wave order, channels stay minor
                    a = a.reshape(perm.size, ch.numel(), 3)[perm].reshape(-1, 3)
                ivs.append(a)
        iv = np.ascontiguousarray(np.concatenate(ivs, 0)) if ivs else np.zeros((0, 3), np.int32)
        buf = np.empty(iv.shape[0] * 3 + 64, dtype=np.uint8)
        n_out = C.c_int64()
        check(lib.masic_range_encode(iv.ctypes.data, iv.shape[0], buf.ctypes.data, buf.size, C.byref(n_out)),
              "masic_range_encode")
        with open(output2, "wb") as f:
            f.write(bytes([order]))
            f.write(buf[:n_out.value].tobytes())
        end = time.time()
        n_symbols = int(iv.shape[0])
        ideal_bits = float(-(np.log2(iv[:, 1].astype(np.float64) / iv[:, 2])).sum()) if iv.shape[0] else 0.0
    num_pixels = pad.h * pad.w * 2
    size1, size2 = os.path.getsize(output1), os.path.getsize(output2)
    return {
        "bpp_real": (size1 + size2) * 8 / num_pixels, "bpp_side": size1 * 8 / num_pixels, "enctime": end - start,
        "y1_hat": out["y1_hat"].clone(), "y2_hat": out["y2_hat"].clone(),
        "z1_hat": out["z1_hat"].clone(), "z2_hat": out["z2_hat"].clone(),
        "y_bits_ideal": ideal_bits, "y_bytes": size2 - 1, "n_symbols": n_symbols, "y_order": y_order,
    }


def _decode_view(eng: HSICEngine, tag: str, dec, flag: np.ndarray, minmax: int) -> torch.Tensor:
    """Sequential (raster) decode of one view's latents; returns y_hat NCHW fp32 and fills eng.buf[tag.y_rnd]."""
    lib = eng.lib
    M, K = eng.M, eng.K
    h16, w16 = eng.H // 16, eng.W // 16
    pm = _PixelModel(eng, tag)
    gmm_in = eng.buf[f"{tag}.gmm_in"]
    ypad = torch.zeros(1, h16 + 4, w16 + 4, M, dtype=ACT, device=eng.dev)
    y_nhwc = torch.zeros(1, h16, w16, M, dtype=torch.float32, device=eng.dev)
    ch_np = np.flatnonzero(flag).astype(np.int32)
    n_ch = int(ch_np.size)
    if n_ch:
        ch = torch.from_numpy(ch_np).to(eng.dev)
        ch_long = ch.long()
        L1 = 2 * minmax + 2
        rows = torch.empty(n_ch, L1, dtype=torch.int32, device=eng.dev)
        rows_h = torch.empty(n_ch, L1, dtype=torch.int32).pin_memory()
        sym_h = np.empty(n_ch, dtype=np.int32)
        for h in range(h16):
            for w in range(w16):
                sig, mu, wl = pm.params_at(ypad, gmm_in, h, w)
                check(lib.masic_gmm_symbol_cdfs(sig.data_ptr(), mu.data_ptr(), wl.data_ptr(), 1, M, K, 1, ch.data_ptr(),
                                                n_ch, minmax, SCALE_BOUND, None, rows.data_ptr(), None, _stream()),
                      "masic_gmm_symbol_cdfs")
                rows_h.copy_(rows)                       # synchronises the pixel's kernels
                check(lib.masic_range_decode_rows(dec, rows_h.data_ptr(), n_ch, L1, sym_h.ctypes.data),
                      "masic_range_decode_rows")
                vals = torch.from_numpy(sym_h.astype(np.float32) - float(minmax)).to(eng.dev)
                y_nhwc[0, h, w, ch_long] = vals
                ypad[0, h + 2, w + 2, ch_long] = vals.to(ACT)
    eng.buf[f"{tag}.y_rnd"].copy_(ypad[:, 2:-2, 2:-2, :])
    return y_nhwc.permute(0, 3, 1, 2).contiguous()


def _decode_view_wave(eng: HSICEngine, tag: str, dec, flag: np.ndarray, minmax: int) -> torch.Tensor:
    """Wavefront decode of one view's latents (positions of wave t = w + 3h in one batch); returns y_hat NCHW fp32 and
    fills eng.buf[tag.y_rnd]."""
    lib = eng.lib
    M, K = eng.M, eng.K
    h16, w16 = eng.H // 16, eng.W // 16
    waves = wave_schedule(h16, w16)
    n_max = max(hs.size for hs, _ in waves)
    cache = eng.__dict__.setdefault("_wave_models", {})          # plans and buffers survive across decompress() calls
    wm = cache.get(tag)
    if wm is None:
        wm = cache[tag] = _WaveModel(eng, tag, n_max)
    gmm_flat = eng.buf[f"{tag}.gmm_in"].view(h16 * w16, -1)
    ypad = torch.zeros(1, h16 + 4, w16 + 4, M, dtype=ACT, device=eng.dev)
    ypad_flat = ypad.view(-1, M)
    y_nhwc = torch.zeros(1, h16, w16, M, dtype=torch.float32, device=eng.dev)
    y_flat = y_nhwc.view(-1, M)
    ch_np = np.flatnonzero(flag).astype(np.int32)
    n_ch = int(ch_np.size)
    if n_ch:
        ch = torch.from_numpy(ch_np).to(eng.dev)
        ch_long = ch.long()
        L1 = 2 * minmax + 2
        rows = torch.empty(n_max * n_ch, L1, dtype=torch.int32, device=eng.dev)
        rows_h = torch.empty(n_max * n_ch, L1, dtype=torch.int32).pin_memory()
        sym_h = torch.empty(n_max * n_ch, dtype=torch.int32).pin_memory()
        # index tensors of every wave, built once on the host
        dy, dx = np.meshgrid(np.arange(5), np.arange(5), indexing="ij")
        sched = []
        for hs, ws in waves:
            crop = ((hs[:, None, None] + dy[None]) * (w16 + 4) + ws[:, None, None] + dx[None]).reshape(-1)
            sched.append((hs.size, crop, hs * w16 + ws, (hs + 2) * (w16 + 4) + ws + 2))
        cat = lambda i: torch.from_numpy(np.concatenate([s_[i] for s_ in sched])).to(eng.dev)   # noqa: E731
        crop_all, pos_all, pad_all = cat(1), cat(2), cat(3)
        c0 = p0 = 0
        for n, crop_i, _, _ in sched:
            crop_idx, pos, pad = crop_all[c0:c0 + crop_i.size], pos_all[p0:p0 + n], pad_all[p0:p0 + n]
            c0 += crop_i.size
            p0 += n
            sig, mu, wl = wm.params_at(ypad_flat, gmm_flat, crop_idx, pos)
            check(lib.masic_gmm_symbol_cdfs(sig.data_ptr(), mu.data_ptr(), wl.data_ptr(), 1, M, K, n, ch.data_ptr(),
                                            n_ch, minmax, SCALE_BOUND, None, rows.data_ptr(), None, _stream()),
                  "masic_gmm_symbol_cdfs")
            rows_h[:n * n_ch].copy_(rows[:n * n_ch])            # synchronises the wave's kernels
            check(lib.masic_range_decode_rows(dec, rows_h.data_ptr(), n * n_ch, L1, sym_h.data_ptr()),
                  "masic_range_decode_rows")
            vals = (sym_h[:n * n_ch].to(eng.dev, non_blocking=True).float() - float(minmax)).view(n, n_ch)
            y_flat[pos[:, None], ch_long[None, :]] = vals
            ypad_flat[pad[:, None], ch_long[None, :]] = vals.to(ACT)
    eng.buf[f"{tag}.y_rnd"].copy_(ypad[:, 2:-2, 2:-2, :])
    return y_nhwc.permute(0, 3, 1, 2).contiguous()


def _wave_tables(eng: HSICEngine):
    """(h, w) of every position in wave order as an int32 device tensor, and the waves' sizes (cached on the engine)."""
    cache = eng.__dict__.setdefault("_wave_tables", None)
    if cache is None:
        h16, w16 = eng.H // 16, eng.W // 16
        waves = wave_schedule(h16, w16)
        hw = np.concatenate([np.stack([hs, ws], 1) for hs, ws in waves]).astype(np.int32)
        cache = eng.__dict__["_wave_tables"] = (torch.from_numpy(np.ascontiguousarray(hw)).to(eng.dev),
                                                 [int(hs.size) for hs, _ in waves])
    return cache


def _decode_view_pairs(eng: HSICEngine, tag: str, table: np.ndarray, data: bytes, lens: np.ndarray) -> torch.Tensor:
    """Wavefront decode of one view of every pair with the range decoder ON THE DEVICE (payload format 2: one stream per
    (pair, non-zero channel), table (3, S) pair | channel | minmax, pair-major like the streams in data).  All pairs
    share the wave schedule: position i of pair b is row b * n_max + i of the static conv plans, so per wave there is
    one gather kernel, the context conv, the parameter nets, one CDF-row kernel and one decode kernel for the whole
    batch (csrc/ydecode.cu).  Returns y_hat NCHW fp32 and fills eng.buf[tag.y_rnd]."""
    lib = eng.lib
    B, M, K = eng.B, eng.M, eng.K
    h16, w16 = eng.H // 16, eng.W // 16
    pos_dev, sizes = _wave_tables(eng)
    n_max = max(sizes)
    cache = eng.__dict__.setdefault("_wave_models", {})
    wm = cache.get(tag)
    if wm is None:
        wm = cache[tag] = _WaveModel(eng, tag, B * n_max)
    gmm_in = eng.buf[f"{tag}.gmm_in"]
    cin = wm.cin
    ypad = torch.zeros(B, h16 + 4, w16 + 4, M, dtype=ACT, device=eng.dev)
    y_nhwc = torch.zeros(B, h16, w16, M, dtype=torch.float32, device=eng.dev)
    S = table.shape[1]
    if S:
        max_minmax = int(table[2].max())
        pitch = 2 * max_minmax + 2
        tab = torch.from_numpy(table).to(eng.dev)
        rows = torch.empty(n_max * S * pitch, dtype=torch.int32, device=eng.dev)
        data_d = torch.frombuffer(bytearray(data), dtype=torch.uint8).to(eng.dev)
        lens_d = torch.from_numpy(lens).to(eng.dev)
        offs = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).to(eng.dev)
        state = torch.zeros(S, 4, dtype=torch.int32, device=eng.dev)
        err = torch.zeros(1, dtype=torch.int32, device=eng.dev)
        check(lib.masic_range_streams_init(data_d.data_ptr(), offs.data_ptr(), S, state.data_ptr(), _stream()),
              "masic_range_streams_init")
        mw = eng.mask_weights.data_ptr() if wm.right else None
        rs = wm.rs.data_ptr() if wm.right else None
        f16 = int(ACT == torch.float16)
        # the loop below issues ~6500 launches at full size, the same for any number of pairs: every pointer and the
        # stream are resolved once, and the status codes are OR-ed and checked after the loop (the host side of the
        # loop is what bounds the decode time)
        st = _stream()
        p_ypad, p_gmm, p_crop, p_px, p_ctx = (t.data_ptr() for t in (ypad, gmm_in, wm.crop, wm.px_in, wm.ctx_out))
        p_sig, p_mu, p_wl, p_rows = (t.data_ptr() for t in (wm.sig, wm.mu, wm.wl, rows))
        p_pair, p_ch, p_mm = (tab[i].data_ptr() for i in range(3))
        p_state, p_data, p_offs, p_y, p_err, p_pos = (t.data_ptr() for t in (state, data_d, offs, y_nhwc, err, pos_dev))
        plan_handles = [wm.ctx_plan._h] + [p._h for p in wm.tail]
        launch = lib.masic_conv_plan_launch
        gather, center, cdfs, decode = (lib.masic_wave_gather_pairs, lib.masic_wave_center,
                                        lib.masic_gmm_symbol_cdfs_pairs, lib.masic_range_decode_wave_pairs)
        off, rc = 0, 0
        for n in sizes:
            pp = p_pos + off * 8
            rc |= gather(p_ypad, h16, w16, M, p_gmm, cin, 2 * M, 4 * M, mw, pp, n, B, n_max, p_crop, rs, p_px, st)
            rc |= launch(plan_handles[0], st)
            rc |= center(p_ctx, cin, 2 * M, 2 * M, B * n_max, p_px, st)
            for h in plan_handles[1:]:
                rc |= launch(h, st)
            rc |= cdfs(p_sig, p_mu, p_wl, 1, M, K, n, n_max, p_pair, p_ch, p_mm, S, max_minmax, SCALE_BOUND, None,
                       p_rows, pitch, None, st)
            rc |= decode(p_rows, n, S, pitch, p_state, p_data, p_offs, p_pair, p_ch, p_mm, max_minmax, pp, h16, w16, M,
                         p_y, p_ypad, f16, p_err, st)
            off += n
        check(rc, "wavefront decode (masic_wave_gather_pairs / conv plans / masic_gmm_symbol_cdfs_pairs / "
                  "masic_range_decode_wave_pairs)")
        # a valid stream ends exactly where the decoder's last renormalisation leaves it (5 + one byte per renormalisation,
        # as the encoder wrote it); a corrupt one almost never does
        bad = torch.stack([err[0], (state[:, 2].long() != lens_d).sum().int()]).cpu()
        if int(bad.abs().sum()):
            raise MasicError("y payload: corrupt range-coded stream")
    eng.buf[f"{tag}.y_rnd"].copy_(ypad[:, 2:-2, 2:-2, :])
    return y_nhwc.permute(0, 3, 1, 2).contiguous()


def _parse_header(header: bytes, M: int):
    """`<name>.npz` -> H, W, [(z string, minmax, non-zero-channel bitmap)] of the two views."""
    def take(n):
        nonlocal p
        if p + n > len(header):
            raise MasicError("header: truncated")
        p += n
        return header[p - n:p]
    p = 0
    H, W = (int(v) for v in np.frombuffer(take(4), dtype=np.uint16))
    views = []
    for _ in range(2):
        length, minmax = (int(v) for v in np.frombuffer(take(4), dtype=np.uint16))
        flag = np.unpackbits(np.frombuffer(take(M // 8), dtype=np.uint8))
        views.append((take(length), minmax, flag))
    return H, W, views


def _header_padding(H: int, W: int) -> Padding:
    """The padded frame of a header's pair size; a size no encoder writes is a corrupt header."""
    try:
        pad = padding_for(H, W)
        pad.check_header()
    except ValueError as e:
        raise MasicError(f"header: {e}") from None
    return pad


def _parse_payload(payload: bytes, hdr):
    """Format-2 `<name>.bin` -> per view (lens int64 (n_ch,), stream bytes), checked against the header's bitmaps."""
    if not payload or payload[0] != ORDER_WAVE_STREAMS:
        raise MasicError("y payload: not format 2 (one range-coded stream per channel); formats 0 and 1 are decoded "
                         "one pair at a time by HSIC.decompress")
    views, p = [], 1
    for _, minmax, flag in hdr:
        if p + 4 > len(payload):
            raise MasicError("y payload: truncated")
        n_ch = int(np.frombuffer(payload[p:p + 4], dtype=np.uint32)[0])
        if n_ch != int(flag.sum()) or (n_ch and minmax < 1):
            raise MasicError("y payload: the stream table does not match the header's non-zero-channel bitmap")
        if p + 4 + 4 * n_ch > len(payload):
            raise MasicError("y payload: truncated")
        lens = np.frombuffer(payload[p + 4:p + 4 + 4 * n_ch], dtype=np.uint32).astype(np.int64)
        p += 4 + 4 * n_ch
        views.append((lens, payload[p:p + int(lens.sum())]))
        p += int(lens.sum())
    if p != len(payload):
        raise MasicError("y payload: its length does not match the stream table")
    return views


def _side_information(model, eng: HSICEngine, pad: Padding, hdrs, h_matrix: torch.Tensor) -> None:
    """Homography products, mask weights and the hyper-synthesis parameters of every pair (MASIC.py:1190-1196,
    :1310-1312) from the z strings of the headers.  The homography is taken to the padded frame of `pad`."""
    o = eng.out
    z_shape = (eng.H // 64, eng.W // 64)
    if pad.aligned:
        eng.Hm.copy_(h_matrix.reshape(eng.B, 3, 3).to(eng.dev))
    else:
        pad.homography_into(_f32c(h_matrix.reshape(eng.B, 3, 3).to(eng.dev)), eng.Hm)
    eng.run_steps(lambda n: n.startswith("warp.prepare") or n.startswith("mask_") or n.startswith("mask2weights"))
    for v, (tag, eb) in enumerate((("L", model.entropy_bottleneck1), ("R", model.entropy_bottleneck2))):
        # one string per call: the reference's EntropyBottleneck.decompress takes batch-1 medians
        z_hat = torch.cat([eb.decompress([h[v][0]], z_shape) for h in hdrs]).to(eng.dev)
        o["z1_hat" if tag == "L" else "z2_hat"].copy_(z_hat)
        eng.buf[f"{tag}.zq"].copy_(z_hat.permute(0, 2, 3, 1))
        eng.run_steps(lambda n, t=tag: n.startswith(f"{t}.h_s."))


def _tail_left(eng: HSICEngine) -> None:
    # left reconstruction, its warp, encoder1 on it and the mask-weighted prior term (:1303-1318)
    eng.run_steps(lambda n: n.startswith("L.g_s.") or n == "R.warp(x1_hat)"
                  or n.startswith("R.g_a(enc1 on warped x1_hat)") or n.startswith("R.y1warp"))


def _tail_right(eng: HSICEngine) -> None:
    eng.run_steps(lambda n: n.startswith("R.g_s.") or n.startswith("R.after_"))


def _decode_pairs(eng: HSICEngine, hdrs, payloads) -> None:
    """y of every pair from format-2 payloads, then both reconstructions; fills eng.out."""
    o = eng.out
    for v, (tag, key) in enumerate((("L", "y1_hat"), ("R", "y2_hat"))):
        flags = np.stack([h[v][2] for h in hdrs]).astype(np.int64)
        minmax = np.array([h[v][1] for h in hdrs], dtype=np.int64)
        table = _stream_table(flags, minmax)
        data = b"".join(p[v][1] for p in payloads)
        lens = np.concatenate([p[v][0] for p in payloads]) if payloads else np.zeros(0, np.int64)
        o[key].copy_(_decode_view_pairs(eng, tag, table, data, lens))
        (_tail_left if tag == "L" else _tail_right)(eng)


def _outputs(o, pad: Padding) -> Dict:
    """The decoded pair cropped to its own size, the latents on the padded grid (as HSIC.forward returns them)."""
    return {k: (pad.crop(o[k]) if k in ("x1_hat", "x2_hat") else o[k]).clone()
            for k in ("x1_hat", "x2_hat", "y1_hat", "y2_hat", "z1_hat", "z2_hat")}


def decompress_batch(model, items, h_matrix: torch.Tensor, device=None) -> Dict:
    """Decode B pairs of one size at once from (header, payload) byte strings in format 2 (what `compress_batch`
    returns, or the `<name>.npz` / `<name>.bin` files `compress` writes).  h_matrix: (B, 3, 3).  Returns x1_hat, x2_hat,
    y1_hat, y2_hat, z1_hat, z2_hat, batched in the order of items and bit-identical to `decompress` of each pair."""
    if model.training:
        raise MasicError("HSIC.decompress_batch: eval mode only")
    items = list(items)
    if not items:
        raise ValueError("HSIC.decompress_batch: no pairs")
    M = model.M
    hdrs, sizes = [], set()
    for header, _ in items:
        H, W, views = _parse_header(bytes(header), M)
        hdrs.append(views)
        sizes.add((H, W))
    if len(sizes) != 1:
        raise ValueError(f"HSIC.decompress_batch: all pairs must share H, W; got {sorted(sizes)}")
    H, W = sizes.pop()
    payloads = [_parse_payload(bytes(payload), hdr) for (_, payload), hdr in zip(items, hdrs)]
    B = len(items)
    if h_matrix.numel() != 9 * B:
        raise ValueError(f"HSIC.decompress_batch: h_matrix must hold {B} homographies, got {tuple(h_matrix.shape)}")
    dev = torch.device(device) if device is not None else h_matrix.device
    if dev.type != "cuda":
        raise MasicError("HSIC.decompress_batch needs a CUDA device: masic_b200 has no CPU fallback")
    pad = _header_padding(H, W)
    eng: HSICEngine = model.engine_for(B, pad.hp, pad.wp, dev)
    with torch.cuda.device(eng.dev):
        _side_information(model, eng, pad, hdrs, h_matrix)
        _decode_pairs(eng, hdrs, payloads)
        return _outputs(eng.out, pad)


def decompress(model, x1: Optional[torch.Tensor], x2: Optional[torch.Tensor], h_matrix: torch.Tensor, output_name,
               output_path: str = "", device=None) -> Dict:
    """HSIC.decompress (MASIC.py:1161-1408).  x1 / x2 are only consulted for the device (the reference uses them
    for shapes, :1313); everything else comes from the two files and the homography."""
    if model.training:
        raise MasicError("HSIC.decompress: eval mode only")
    lib = _lib.load()
    output1 = os.path.join(output_path, str(output_name) + ".npz")
    output2 = os.path.join(output_path, str(output_name) + ".bin")
    with open(output1, "rb") as f:
        H, W, hdr = _parse_header(f.read(), model.M)
    dev = h_matrix.device if device is None else torch.device(device)
    if dev.type != "cuda":
        dev = x1.device if x1 is not None else torch.device("cuda:0")
    pad = _header_padding(H, W)
    eng: HSICEngine = model.engine_for(1, pad.hp, pad.wp, dev)
    o = eng.out
    with torch.cuda.device(eng.dev):
        _side_information(model, eng, pad, [hdr], h_matrix)
        with open(output2, "rb") as f:
            raw = f.read()
        if not raw or raw[0] not in (ORDER_RASTER, ORDER_WAVE, ORDER_WAVE_STREAMS):
            raise MasicError(f"{output2}: unknown symbol-order tag in the y payload")
        if raw[0] == ORDER_WAVE_STREAMS:
            payload = _parse_payload(raw, hdr)
            start = time.time()
            _decode_pairs(eng, [hdr], [payload])
            torch.cuda.synchronize(eng.dev)
            end = time.time()
        else:
            decode_view = _decode_view_wave if raw[0] == ORDER_WAVE else _decode_view
            data = np.frombuffer(raw, dtype=np.uint8)[1:].copy()
            dec = C.c_void_p()
            check(lib.masic_range_decoder_create(data.ctypes.data, data.size, C.byref(dec)), "masic_range_decoder_create")
            try:
                start = time.time()
                o["y1_hat"].copy_(decode_view(eng, "L", dec, hdr[0][2], hdr[0][1]))
                _tail_left(eng)
                o["y2_hat"].copy_(decode_view(eng, "R", dec, hdr[1][2], hdr[1][1]))
                _tail_right(eng)
                torch.cuda.synchronize(eng.dev)
                end = time.time()
            finally:
                lib.masic_range_decoder_destroy(dec)
        outputs = _outputs(o, pad)
    return {**outputs, "dectime": end - start}
