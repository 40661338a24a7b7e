"""HSICEngine — the B200-native execution plan of MASIC's codec forward pass.

Restates *what* coremasic/mywork/MASIC.py:744-851 (HSIC.forward, eval mode) computes as a
fixed sequence of hand-written CUDA kernels over pre-allocated HBM buffers:

  * activations live in NHWC bf16 (fp32 for latents, entropy parameters and images);
  * every 5x5 / 3x3 / 1x1 conv and stride-2 transposed conv is one tcgen05 implicit-GEMM
    launch (masic_b200/csrc/conv_tc.cu) with bias, ReLU/LeakyReLU, GDN/IGDN and the
    mask-weight scaling fused into its epilogue; concatenations are free (layers write
    into channel slices of a shared buffer);
  * the three 1x1 entropy-parameter branches share one wide GEMM for their first layer;
  * warp, masks, pre/after convs, likelihoods and quantisation are fused memory-bound kernels;
  * duplicated work in the reference (warp of x1_hat at :821 and :833, round(y1) at :755
    and :767) is computed once;
  * the whole sequence is captured in a CUDA graph and replayed per stereo pair.

The engine is built for a fixed (batch, H, W); H and W must be multiples of 64
(MASIC.py:1191-1192).  It never touches the CPU: there is no fallback path.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import _lib, ops
from ._lib import MasicError, check
from .convplan import (ACT_LEAKY, ACT_NONE, ACT_RELU, CONV, CONV_XFOLD8, DECONV_S2, GDN_FWD, GDN_INV,
                       GDN_NONE, MASK_A_5x5, ConvPlan, DeconvImgPlan, PackedConv, fold8_weights_5x5_s1)

F16 = _lib.FMT_F16              # the inference engines run on fp16 operands / activations (csrc/cvt16.cuh)
ACT = _lib.act_dtype(F16)
SCALE_BOUND = 0.11
IMG_CP = 8           # channel pitch of the 16-bit images feeding g_a_conv1 (3 real channels, stored split: [hi | lo]);
XOFF, XPAD = _lib.IMG_XOFF, _lib.IMG_XPAD   # rows padded: [N][H][W+XPAD][8], pixel x at column x+XOFF (XFOLD8 input)


class HSICEngine:
    def __init__(self, sd: Dict[str, torch.Tensor], batch: int, height: int, width: int,
                 device: torch.device | str = "cuda:0", N: int = 128, M: int = 192, K: int = 5,
                 use_graph: bool = True):
        if height % 64 or width % 64:
            raise ValueError("HSIC needs H and W to be multiples of 64 (y = x/16, z = y/4)")
        if (N, M, K) != (128, 192, 5):
            raise MasicError("the sm_100a kernels are specialised for HSIC(N=128, M=192, K=5) "
                             "(MASIC.py:653; the only configuration the reference scripts use)")
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("HSICEngine runs on a CUDA device only (no CPU fallback)")
        self.B, self.H, self.W, self.N, self.M, self.K = batch, height, width, N, M, K
        self.sd = {k: v.detach().to(self.dev) for k, v in sd.items()}
        self.steps: List[Tuple[str, Callable[[], None]]] = []      # kernel launches, issue order
        self.sched: List[Tuple] = []     # ("run", idx, lane) | ("record", key, lane) | ("wait", key, lane)
        self._lane = 0
        self.plans: Dict[str, ConvPlan] = {}
        self.buf: Dict[str, torch.Tensor] = {}     # named internal buffers (bitstream.py drives partial runs)
        self.packs: Dict[str, PackedConv] = {}     # packed weights the per-pixel decoder re-uses
        self._keep = []
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.use_graph = use_graph
        with torch.cuda.device(self.dev):
            self._build()

    # ------------------------------------------------------------------ helpers
    def _buf(self, *shape, dtype=ACT):
        return torch.zeros(*shape, dtype=dtype, device=self.dev)

    def _w(self, name):
        return self.sd[name].float().contiguous()

    def _add(self, name: str, fn: Callable[[], None]):
        self.steps.append((name, fn))
        self.sched.append(("run", len(self.steps) - 1, self._lane))

    # Three lanes (CUDA streams) inside the captured graph: lane 0 carries the critical path
    # (encoder1 -> decoder1 -> warp -> encoder1 again -> gmm2 -> decoder2), lane 1 the left view's
    # hyper/context/GMM chain, lane 2 the right view's encoder + hyper chain and the mask chain.
    # Most of lanes 1/2 are small launches (<= 148 work items) that would otherwise leave SMs idle.
    def _on(self, lane: int):
        self._lane = lane

    def _record(self, key: str):
        self.sched.append(("record", key, self._lane))

    def _wait(self, key: str):
        self.sched.append(("wait", key, self._lane))

    def _s(self):
        return torch.cuda.current_stream().cuda_stream

    def _conv(self, name: str, packed: PackedConv, x, out, *, stride=1, tap_mask=0, in_coff=0, out_coff=0,
              act=ACT_NONE, rowscale=None, rs_off=0, cta_pairs=False):
        plan = ConvPlan(packed=packed, stride=stride, tap_mask=tap_mask, x=x, in_coff=in_coff, out=out,
                        out_coff=out_coff, act=act, rowscale=rowscale, rs_off=rs_off, cta_pairs=cta_pairs)
        self.plans[name] = plan
        self._add(name, plan.launch)
        return plan

    def _pack(self, prefix: str, *, kind=CONV, ksize=5, c_in, c_out, n_tile, transposed=False, gdn=GDN_NONE,
              gdn_prefix=None, c_out_pad=None, pad_cin_from=None):
        w = self._w(prefix + ".weight")
        if pad_cin_from is not None:                      # g_a_conv1: 3 -> IMG_CP input channels
            wp = torch.zeros(w.shape[0], c_in, w.shape[2], w.shape[3], device=self.dev)
            wp[:, :pad_cin_from] = w
            w = wp
        return PackedConv(kind=kind, ksize=ksize, c_in=c_in, c_out=c_out, n_tile=n_tile, weight=w,
                          transposed=transposed, bias=self._w(prefix + ".bias"), c_out_pad=c_out_pad, gdn=gdn,
                          gdn_beta=self._w(gdn_prefix + ".beta") if gdn else None,
                          gdn_gamma=self._w(gdn_prefix + ".gamma") if gdn else None, f16=F16)

    # ------------------------------------------------------------------ building blocks
    def _encoder_weights(self, enc: str):
        N, M = self.N, self.M
        return [
            self._pack(f"{enc}.g_a_conv1", kind=CONV_XFOLD8, c_in=64, c_out=N, n_tile=128, gdn=GDN_FWD,
                       gdn_prefix=f"{enc}.g_a_gdn1"),
            self._pack(f"{enc}.g_a_conv2", c_in=N, c_out=N, n_tile=128, gdn=GDN_FWD, gdn_prefix=f"{enc}.g_a_gdn2"),
            self._pack(f"{enc}.g_a_conv3", c_in=N, c_out=N, n_tile=128, gdn=GDN_FWD, gdn_prefix=f"{enc}.g_a_gdn3"),
            self._pack(f"{enc}.g_a_conv4", c_in=N, c_out=M, n_tile=192),
        ]

    def _encoder(self, tag: str, packs, img_bf16):
        """g_a: 4x (conv5 s2 [+GDN]) — MASIC.py:521-531.  Returns the fp32 NHWC latent."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        e1 = self._buf(B, H // 2, W // 2, N)
        e2 = self._buf(B, H // 4, W // 4, N)
        e3 = self._buf(B, H // 8, W // 8, N)
        y = self._buf(B, H // 16, W // 16, M, dtype=torch.float32)
        self._conv(f"{tag}.conv1+gdn", packs[0], img_bf16, e1, stride=2)
        # CTA pairs (cta_group::2) measured faster on these two, the wide 1x1 / 3x3 layers and the context conv only
        self._conv(f"{tag}.conv2+gdn", packs[1], e1, e2, stride=2, cta_pairs=True)
        self._conv(f"{tag}.conv3+gdn", packs[2], e2, e3, stride=2, cta_pairs=True)
        self._conv(f"{tag}.conv4", packs[3], e3, y, stride=2)
        return y

    def _decoder(self, tag: str, dec: str, yq_bf16, out_img, igdn_prefix=None, out16=None):
        """g_s: 3x (deconv5 s2 + IGDN) + deconv5 s2 -> 3 — MASIC.py:544-554.  The last layer runs in col2im form
        (csrc/deconv_img.cu) and writes the NCHW fp32 image `out_img`, with after_gdn fused for the right view."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        g1 = self._buf(B, H // 8, W // 8, N)
        g2 = self._buf(B, H // 4, W // 4, N)
        g3 = self._buf(B, H // 2, W // 2, N)
        p1 = self._pack(f"{dec}.g_s_conv1", kind=DECONV_S2, c_in=M, c_out=N, n_tile=128, transposed=True,
                        gdn=GDN_INV, gdn_prefix=f"{dec}.g_s_gdn1")
        p2 = self._pack(f"{dec}.g_s_conv2", kind=DECONV_S2, c_in=N, c_out=N, n_tile=128, transposed=True,
                        gdn=GDN_INV, gdn_prefix=f"{dec}.g_s_gdn2")
        p3 = self._pack(f"{dec}.g_s_conv3", kind=DECONV_S2, c_in=N, c_out=N, n_tile=128, transposed=True,
                        gdn=GDN_INV, gdn_prefix=f"{dec}.g_s_gdn3")
        self._conv(f"{tag}.deconv1+igdn", p1, yq_bf16, g1)
        self._conv(f"{tag}.deconv2+igdn", p2, g1, g2)
        self._conv(f"{tag}.deconv3+igdn", p3, g2, g3)
        ib = self._w(igdn_prefix + ".beta") if igdn_prefix else None
        ig = self._w(igdn_prefix + ".gamma") if igdn_prefix else None
        plan = DeconvImgPlan(x=g3, weight=self._w(f"{dec}.g_s_conv4.weight"), bias=self._w(f"{dec}.g_s_conv4.bias"),
                             out=out_img, igdn_beta=ib, igdn_gamma=ig, out16=out16, out16_coff=0, out16_xoff=XOFF)
        self.plans[f"{tag}.deconv4(col2im)"] = plan
        self._add(f"{tag}.deconv4(col2im)", plan.launch)

    def _hyper(self, tag: str, idx: int, y_abs_bf16, gmm_in, rowscale=None):
        """h_a -> EntropyBottleneck -> h_s_up (MASIC.py:747-754 / :786-793).  Writes params into
        gmm_in[..., 0:2M].  Returns (z_hat_nchw, z_lik_nchw)."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        h16, w16 = H // 16, W // 16
        ha = f"_h_a{idx}.encode_hyper"
        c1 = self._buf(B, h16, w16, N)
        c2 = self._buf(B, h16 // 2, w16 // 2, N)
        z = self._buf(B, h16 // 4, w16 // 4, N, dtype=torch.float32)
        self._conv(f"{tag}.h_a.conv1", self._pack(f"{ha}.0", c_in=M, c_out=N, n_tile=128), y_abs_bf16, c1,
                   stride=1, act=ACT_RELU)
        # 27 and 10 spatial tiles only: narrow n-tiles spread them over 108 / 40 CTAs (a lone CTA streaming 50 k-blocks is
        # bound by one SM's L2 bandwidth; tools/conv_perf.py mb_ha2 / mb_ha3: 0.026 -> 0.022, 0.025 -> 0.021 ms)
        self._conv(f"{tag}.h_a.conv2", self._pack(f"{ha}.2", c_in=N, c_out=N, n_tile=32), c1, c2, stride=2,
                   act=ACT_RELU)
        self._conv(f"{tag}.h_a.conv3", self._pack(f"{ha}.4", c_in=N, c_out=N, n_tile=32), c2, z, stride=2)
        # EntropyBottleneck (entropy_models.py:384-411)
        eb = f"entropy_bottleneck{idx}."
        mats = [self._w(f"{eb}_matrices.{i}") for i in range(5)]
        bias = [self._w(f"{eb}_biases.{i}") for i in range(5)]
        facs = [self._w(f"{eb}_factors.{i}") for i in range(4)]
        quant = self._w(f"{eb}quantiles")
        self._keep += [mats, bias, facs, quant]
        pm = (C.c_void_p * 5)(*[t.data_ptr() for t in mats])
        pb = (C.c_void_p * 5)(*[t.data_ptr() for t in bias])
        pf = (C.c_void_p * 4)(*[t.data_ptr() for t in facs])
        hw64 = (h16 // 4) * (w16 // 4)
        z_hat = self._buf(B, N, h16 // 4, w16 // 4, dtype=torch.float32)
        z_lik = self._buf(B, N, h16 // 4, w16 // 4, dtype=torch.float32)
        zq = self._buf(B, h16 // 4, w16 // 4, N)
        self.buf[f"{tag}.z"], self.buf[f"{tag}.zq"] = z, zq

        def eb_step():
            check(self.lib.masic_eb_fwd(z.data_ptr(), 1, B, N, hw64, pm, pb, pf, quant.data_ptr(), z_hat.data_ptr(),
                                        z_lik.data_ptr(), None, 0, zq.data_ptr(), N, F16, self._s()), "masic_eb_fwd")
        self._add(f"{tag}.entropy_bottleneck", eb_step)
        # h_s_up: deconv5 s2 -> LeakyReLU -> deconv5 s2 -> LeakyReLU -> conv3 s1 (MASIC.py:678-691)
        hs = f"h_s{idx}_up"
        d1 = self._buf(B, h16 // 2, w16 // 2, M)
        d2 = self._buf(B, h16, w16, 2 * M)                   # 288 real channels, 384 pitch (zeros beyond)
        self._conv(f"{tag}.h_s.deconv1", self._pack(f"{hs}.0", kind=DECONV_S2, c_in=N, c_out=M, n_tile=192,
                                                      transposed=True), zq, d1, act=ACT_LEAKY)
        self._conv(f"{tag}.h_s.deconv2", self._pack(f"{hs}.2", kind=DECONV_S2, c_in=M, c_out=M * 3 // 2, n_tile=192,
                                                      transposed=True), d1, d2, act=ACT_LEAKY)
        self._conv(f"{tag}.h_s.conv3x3", self._pack(f"{hs}.4", ksize=3, c_in=M * 3 // 2, c_out=2 * M, n_tile=192),
                   d2, gmm_in, stride=1, out_coff=0, rowscale=rowscale, rs_off=0, cta_pairs=True)
        return z_hat, z_lik

    def _gmm_net(self, tag: str, net: str, cin: int, first_is_deconv: bool, gmm_in):
        """Three 1x1 branches (MASIC.py:338-376 / :410-444): layer 0 fused into one wide GEMM.
        Returns fp32 NHWC (sigma, mu, weight-logits), each [B, h16, w16, M*K]."""
        B, H, W, M, K = self.B, self.H, self.W, self.M, self.K
        h16, w16 = H // 16, W // 16
        MK = M * K
        t = first_is_deconv
        cat_dim = 1 if t else 0
        br = ("gmm_sigma", "gmm_means", "gmm_weights")
        w0 = torch.cat([self._w(f"{net}.{b}.0.weight") for b in br], dim=cat_dim)
        b0 = torch.cat([self._w(f"{net}.{b}.0.bias") for b in br])
        p0 = PackedConv(ksize=1, c_in=cin, c_out=18 * M, n_tile=192, weight=w0, transposed=t, bias=b0, f16=F16)
        self.packs[f"{tag}.gmm.l0"] = p0
        l0 = self._buf(B, h16, w16, 18 * M)
        self._conv(f"{tag}.gmm.l0(3 branches)", p0, gmm_in, l0,
                   act=[ACT_RELU] * 6 + [ACT_LEAKY] * 12, cta_pairs=True)
        def pk(b, i, ci, co):
            pc = PackedConv(ksize=1, c_in=ci, c_out=co, n_tile=192, weight=self._w(f"{net}.{b}.{i}.weight"),
                            transposed=t if i == 2 else False, bias=self._w(f"{net}.{b}.{i}.bias"), f16=F16)
            self.packs[f"{tag}.gmm.{b[4:]}.l{i // 2}"] = pc          # per-branch packs: the per-pixel decoder's plans
            return pc

        def mat(b, i):                     # 1x1 weight as (c_out, c_in); layer-1 heads of the y1 net are ConvTranspose2d
            w = self._w(f"{net}.{b}.{i}.weight")[:, :, 0, 0]
            return w.t() if (t and i == 2) else w

        for b_, i_, ci_, co_ in (("gmm_sigma", 2, 6 * M, 4 * M), ("gmm_means", 2, 6 * M, 4 * M),
                                 ("gmm_weights", 2, 6 * M, MK), ("gmm_sigma", 4, 4 * M, MK),
                                 ("gmm_means", 4, 4 * M, MK), ("gmm_weights", 4, MK, MK)):
            pk(b_, i_, ci_, co_)
        # layer 1 of the three branches as ONE grouped launch (block-diagonal: each branch reads its own 6M slice of
        # l0), layer 2 as two (sigma | means share K = 4M; weights has K = 5M): 4 launches per view instead of 7,
        # 1105 / 850 work items instead of 3 x 340-425 (less wave quantisation on 148 SMs)
        nt = lambda c: c // 192
        l1 = self._buf(B, h16, w16, 13 * M)               # sigma 4M | means 4M | weights 5M
        w1 = torch.cat([mat(b_, 2) for b_ in br], dim=0).reshape(13 * M, 6 * M, 1, 1).contiguous()
        b1 = torch.cat([self._w(f"{net}.{b_}.2.bias") for b_ in br])
        p1 = PackedConv(ksize=1, c_in=6 * M, c_out=13 * M, n_tile=192, weight=w1, bias=b1, f16=F16)
        self.packs[f"{tag}.gmm.l1(3 branches)"] = p1            # the wave decoder runs the same grouped launches
        plan = ConvPlan(packed=p1, x=l0, out=l1, act=[ACT_RELU] * nt(4 * M) + [ACT_LEAKY] * nt(9 * M),
                        nt_in_coff=[0] * nt(4 * M) + [6 * M] * nt(4 * M) + [12 * M] * nt(5 * M))
        self.plans[f"{tag}.gmm.l1(3 branches)"] = plan
        self._add(f"{tag}.gmm.l1(3 branches)", plan.launch)
        smw = self._buf(3 * B, h16, w16, MK, dtype=torch.float32)     # sigma | mu | weight logits, each dense [B][P][MK]
        sig, mu, wl = smw[0:B], smw[B:2 * B], smw[2 * B:3 * B]
        w2 = torch.cat([mat("gmm_sigma", 4), mat("gmm_means", 4)], dim=0).reshape(2 * MK, 4 * M, 1, 1).contiguous()
        b2 = torch.cat([self._w(f"{net}.gmm_sigma.4.bias"), self._w(f"{net}.gmm_means.4.bias")])
        p2 = PackedConv(ksize=1, c_in=4 * M, c_out=2 * MK, n_tile=192, weight=w2, bias=b2, f16=F16)
        self.packs[f"{tag}.gmm.l2(sigma|means)"] = p2
        tiles = list(range(0, MK, 192))
        plan = ConvPlan(packed=p2, x=l1, out=smw, act=[ACT_RELU] * nt(MK) + [ACT_NONE] * nt(MK),
                        nt_in_coff=[0] * nt(MK) + [4 * M] * nt(MK), nt_out_coff=tiles + tiles,
                        nt_out_img=[0] * nt(MK) + [B] * nt(MK))
        self.plans[f"{tag}.gmm.l2(sigma|means)"] = plan
        self._add(f"{tag}.gmm.l2(sigma|means)", plan.launch)
        self._conv(f"{tag}.gmm.weights.l2", self.packs[f"{tag}.gmm.weights.l2"], l1, wl, in_coff=8 * M)
        self.buf[f"{tag}.sigma"], self.buf[f"{tag}.mu"], self.buf[f"{tag}.wlogit"] = sig, mu, wl
        return sig, mu, wl

    def _gmm_likelihood(self, tag, y, sig, mu, wl, y_hat_nchw, lik_nchw):
        B, M, K = self.B, self.M, self.K
        hw = y.shape[1] * y.shape[2]

        def step():
            check(self.lib.masic_gmm_likelihood_fwd(y.data_ptr(), sig.data_ptr(), mu.data_ptr(), wl.data_ptr(), 1, 1,
                                                    B, M, K, hw, SCALE_BOUND, y_hat_nchw.data_ptr(), lik_nchw.data_ptr(),
                                                    None, 0, None, 0, 0, None, 0, 0, F16, self._s()),
                  "masic_gmm_likelihood_fwd")
        self._add(f"{tag}.gmm_likelihood", step)

    def _latent_prep(self, tag, y, y_abs, y_rnd, rnd_coff=0, rowscale=None, rs_off=0):
        npix = y.shape[0] * y.shape[1] * y.shape[2]
        c = y.shape[3]

        def step():
            check(self.lib.masic_latent_prep(y.data_ptr(), npix, c, None if y_abs is None else y_abs.data_ptr(),
                                             0 if y_abs is None else y_abs.shape[3],
                                             None if y_rnd is None else y_rnd.data_ptr(),
                                             0 if y_rnd is None else y_rnd.shape[3], rnd_coff,
                                             None if rowscale is None else rowscale.data_ptr(),
                                             0 if rowscale is None else rowscale.shape[3], rs_off, F16, self._s()),
                  "masic_latent_prep")
        self._add(f"{tag}.latent_prep", step)

    # ------------------------------------------------------------------ the plan
    def _build(self):
        B, H, W, N, M, K = self.B, self.H, self.W, self.N, self.M, self.K
        h16, w16 = H // 16, W // 16
        f32 = torch.float32
        # static inputs / outputs (NCHW fp32, the reference's tensor format)
        self.x1 = self._buf(B, 3, H, W, dtype=f32)
        self.x2 = self._buf(B, 3, H, W, dtype=f32)
        self.Hm = torch.eye(3, device=self.dev).repeat(B, 1, 1).contiguous()
        o = self.out = {
            "x1_hat": self._buf(B, 3, H, W, dtype=f32), "x2_hat": self._buf(B, 3, H, W, dtype=f32),
            "y1_hat": self._buf(B, M, h16, w16, dtype=f32), "y2_hat": self._buf(B, M, h16, w16, dtype=f32),
            "x1_mask_R": self._buf(B, 1, H, W, dtype=f32), "x1_mask_L": self._buf(B, 1, H, W, dtype=f32),
            "lik_y1": self._buf(B, M, h16, w16, dtype=f32), "lik_y2": self._buf(B, M, h16, w16, dtype=f32),
        }

        # ---------------- lane 0: left encoder (MASIC.py:746, :755)
        self._on(0)
        x1_bf = self._buf(B, H, W + XPAD, IMG_CP)
        self._add("x1.pack_nhwc", lambda: ops.nchw_to_nhwc_into(self.x1, x1_bf, split=True))
        enc1 = self._encoder_weights("encoder1")
        y1 = self._encoder("L.g_a", enc1, x1_bf)
        y1_abs = self._buf(B, h16, w16, M)
        y1_rnd = self._buf(B, h16, w16, M)
        self._latent_prep("L", y1, y1_abs, y1_rnd)
        self.buf["L.y"], self.buf["L.y_rnd"] = y1, y1_rnd
        self._record("y1")

        # ---------------- lane 2: homography products, mask weights, right encoder + hyper chain
        # (MASIC.py:781-805; none of it depends on the left view's latents)
        self._on(2)
        T = torch.empty(B, 3, 3, device=self.dev, dtype=torch.float64)
        Tinv = torch.empty(B, 3, 3, device=self.dev, dtype=torch.float64)
        self._add("warp.prepare", lambda: (ops.warp_prepare_into(self.Hm, T, (H, W), (H, W)),
                                           ops.warp_prepare_into(self.Hm, Tinv, (H, W), (H, W), invert=True)))
        self._record("T")
        # x1 and the all-ones image are warped by ONE launch (same transform: the fp64 coordinates, ~60 % of the kernel's
        # instructions, are evaluated once)
        x1_warp = self._buf(B, 3, H, W, dtype=f32)
        self._add("R.warp(x1)+mask_R", lambda: ops.warp_perspective_into(self.x1, T, (H, W), dst=x1_warp,
                                                                         ones=o["x1_mask_R"]))
        self._add("mask_L=warp(mask_R,Hinv)", lambda: ops.warp_perspective_into(o["x1_mask_R"], Tinv, (H, W),
                                                                                dst=o["x1_mask_L"]))
        # mask2weights: 4x (conv3 s2 [+ReLU]) + softmax over 3 (MASIC.py:472-506)
        mk = "mask2weights_unit.maskconv"
        mw = self._buf(B, h16, w16, 3, dtype=f32)        # per-pixel fusion weights, NHWC
        self.mask_weights = mw
        mws = [self._w(f"{mk}.{i}.weight") for i in (0, 2, 4, 6)]
        mbs = [self._w(f"{mk}.{i}.bias") for i in (0, 2, 4, 6)]
        self._add("mask2weights(fused)", lambda: ops.mask2weights_into(o["x1_mask_R"], mws, mbs, out_nhwc=mw))
        self._record("mw")
        x2in_bf = self._buf(B, H, W + XPAD, IMG_CP)
        pre_w, pre_b = self._w("encoder2.pre_conv.weight"), self._w("encoder2.pre_conv.bias")
        pre_beta, pre_gamma = self._w("encoder2.pre_gdn.beta"), self._w("encoder2.pre_gdn.gamma")
        self._add("R.pre_conv+pre_gdn", lambda: ops.conv_small_into(
            x1_warp, self.x2, pre_w, pre_b, ksize=5, stride=1, gdn=GDN_FWD, beta=pre_beta, gamma=pre_gamma, out16=x2in_bf,
            split=True))
        y2 = self._encoder("R.g_a", self._encoder_weights("encoder2"), x2in_bf)
        y2_abs = self._buf(B, h16, w16, M)
        y2_rnd = self._buf(B, h16, w16, M)
        self._latent_prep("R", y2, y2_abs, y2_rnd)
        self.buf["R.y"], self.buf["R.y_rnd"] = y2, y2_rnd
        gmm2_in = self._buf(B, h16, w16, 5 * M)
        self.buf["R.gmm_in"] = gmm2_in
        o["z2_hat"], o["lik_z2"] = self._hyper("R", 2, y2_abs, gmm2_in, rowscale=mw)           # params2 * w0
        ctx2 = self._pack("context_prediction2", c_in=M, c_out=2 * M, n_tile=192)
        self.packs["R.context"] = ctx2
        self._conv("R.context(masked5x5)", ctx2, y2_rnd, gmm2_in, stride=1, tap_mask=MASK_A_5x5, out_coff=2 * M,
                   rowscale=mw, rs_off=1, cta_pairs=True)                                                          # ctx2 * w1
        self._record("right")

        # ---------------- lane 1: left hyperprior, context, GMM parameters, likelihood (MASIC.py:747-767)
        self._on(1)
        self._wait("y1")
        gmm1_in = self._buf(B, h16, w16, 4 * M)
        self.buf["L.gmm_in"] = gmm1_in
        o["z1_hat"], o["lik_z1"] = self._hyper("L", 1, y1_abs, gmm1_in)
        ctx1 = self._pack("context_prediction1", c_in=M, c_out=2 * M, n_tile=192)
        self.packs["L.context"] = ctx1
        self._conv("L.context(masked5x5)", ctx1, y1_rnd, gmm1_in, stride=1, tap_mask=MASK_A_5x5, out_coff=2 * M,
                   cta_pairs=True)
        s1, m1, w1 = self._gmm_net("L", "_h_s1_same_resolution", 4 * M, True, gmm1_in)
        self._gmm_likelihood("L", y1, s1, m1, w1, o["y1_hat"], o["lik_y1"])
        self._record("left_entropy")

        # ---------------- lane 0: left decoder, warp of x1_hat, encoder1 on it, right GMM + decoder
        self._on(0)
        self._decoder("L.g_s", "decoder1", y1_rnd, o["x1_hat"])                                    # :777
        # x1_hat warped once (the reference computes it twice, :821 and :833)
        x1hw_bf = self._buf(B, H, W + XPAD, IMG_CP)
        # after_conv on the tensor cores: its two inputs are written straight into ONE channels-last 16-bit image
        # [after_gdn(g_s(y2_hat)) (3) 0 | x1_hat_warp (3) 0], each producer with one aligned 8-byte store per pixel
        ac_in = self._buf(B, H, W + XPAD, IMG_CP)
        self._wait("T")
        self._add("R.warp(x1_hat)", lambda: ops.warp_perspective_into(o["x1_hat"], T, (H, W), dst16=x1hw_bf, split=True,
                                                                      dst2=ac_in, dst2_coff=4))
        y1w = self._encoder("R.g_a(enc1 on warped x1_hat)", enc1, x1hw_bf)                         # :822
        self._wait("mw")
        self._wait("right")
        self._latent_prep("R.y1warp", y1w, None, gmm2_in, rnd_coff=4 * M, rowscale=mw, rs_off=2)   # round(.) * w2
        s2, m2, w2 = self._gmm_net("R", "_h_s2_same_resolution", 5 * M, False, gmm2_in)            # :827
        self._gmm_likelihood("R", y2, s2, m2, w2, o["y2_hat"], o["lik_y2"])                        # :829
        self._decoder("R.g_s", "decoder2", y2_rnd, None, igdn_prefix="decoder2.after_gdn", out16=ac_in)   # :834, :615
        wf, bf_, tmask = fold8_weights_5x5_s1(self._w("decoder2.after_conv.weight"), self._w("decoder2.after_conv.bias"),
                                              transposed=True, slots=(0, 1, 2, 4, 5, 6))
        pk = PackedConv(ksize=5, c_in=64, c_out=48, n_tile=48, weight=wf, bias=bf_, f16=F16)
        self.packs["R.after_conv"] = pk
        plan = ConvPlan(packed=pk, x=ac_in.view(B, H, (W + XPAD) // 8, 64), stride=1, tap_mask=tmask, w_in=W // 8,
                        out=o["x2_hat"].view(B * 3, H, W // 8, 8), out_blk_images=True)
        plan.flops = 2.0 * B * H * W * 6 * 3 * 25         # useful work (the folded GEMM multiplies mostly zeros)
        plan.hbm_bytes = B * H * W * (16.0 + 12.0)
        self.plans["R.after_conv"] = plan
        self._add("R.after_conv", plan.launch)
        self._wait("left_entropy")
        self.flops = sum(p.flops for p in self.plans.values())

    # ------------------------------------------------------------------ running
    def _launch_all(self, concurrent: bool = True):
        """Issue every step.  concurrent=True spreads the three lanes over CUDA streams (fork from the
        current stream, join back into it); False issues everything in order on the current stream."""
        if not concurrent:
            for _, fn in self.steps:
                fn()
            return
        main = torch.cuda.current_stream()
        if getattr(self, "_side", None) is None:
            self._side = [torch.cuda.Stream(device=self.dev), torch.cuda.Stream(device=self.dev)]
        lanes = [main] + self._side
        for sd in self._side:
            sd.wait_stream(main)                       # fork
        events: Dict[str, torch.cuda.Event] = {}
        for kind, a, lane in self.sched:
            if kind == "run":
                with torch.cuda.stream(lanes[lane]):
                    self.steps[a][1]()
            elif kind == "record":
                ev = torch.cuda.Event()
                ev.record(lanes[lane])
                events[a] = ev
            else:
                lanes[lane].wait_event(events[a])
        for sd in self._side:
            main.wait_stream(sd)                       # join

    def run(self, x1: Optional[torch.Tensor] = None, x2: Optional[torch.Tensor] = None,
            h_matrix: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """Run one forward pass.  Inputs (device tensors, NCHW fp32 / (B,3,3)) are copied into
        the static input buffers; the returned dict aliases the static output buffers."""
        with torch.cuda.device(self.dev):
            if x1 is not None:
                self.x1.copy_(x1, non_blocking=True)
            if x2 is not None:
                self.x2.copy_(x2, non_blocking=True)
            if h_matrix is not None:
                self.Hm.copy_(h_matrix.reshape(self.B, 3, 3), non_blocking=True)
            if not self.use_graph:
                self._launch_all()
            else:
                if self.graph is None:
                    self._capture()
                self.graph.replay()
        return self.out

    def _capture(self):
        self._launch_all()                      # warm-up: cudaFuncSetAttribute etc. outside capture
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._launch_all()
        self.graph = g

    def run_steps(self, select: Callable[[str], bool]) -> List[str]:
        """Eagerly issue, in plan order on the current stream, the steps whose name `select` accepts
        (the decoder runs the plan piecewise around its sequential latent decode)."""
        done = []
        with torch.cuda.device(self.dev):
            for name, fn in self.steps:
                if select(name):
                    fn()
                    done.append(name)
        return done

    def profile_steps(self, iters: int = 3) -> List[Tuple[str, float]]:
        """Eager run with a CUDA-event pair around every step; median ms per step.  Every iteration starts with a ~3 ms
        device-side sleep so that the host has enqueued all launches and events before the first kernel runs: the
        events then time the kernels back to back, not the host's launch rate (a step of 10-30 us is shorter than
        one Python launch)."""
        with torch.cuda.device(self.dev):
            self._launch_all(concurrent=False)
            torch.cuda.synchronize()
            acc = [[] for _ in self.steps]
            for _ in range(iters):
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self.steps) + 1)]
                torch.cuda._sleep(6_000_000)
                evs[0].record()
                for i, (_, fn) in enumerate(self.steps):
                    fn()
                    evs[i + 1].record()
                torch.cuda.synchronize()
                for i in range(len(self.steps)):
                    acc[i].append(evs[i].elapsed_time(evs[i + 1]))
            return [(self.steps[i][0], sorted(a)[len(a) // 2]) for i, a in enumerate(acc)]
