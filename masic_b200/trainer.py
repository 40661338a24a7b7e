"""HSICTrainer — MASIC's codec TRAINING STEP on the B200-native kernels (BASELINE.json configs[4]).

Restates what one iteration of coremasic/mywork/newtrain_codec_real.py:105-146 computes:

    out  = HSIC.forward(x1, x2, h)  in train() mode        MASIC.py:744-851 ('noise' quantisation)
    loss = lambda * 255^2 * (mse1 + mse2) + bpp            newtrain_codec_real.py:66-87
    loss.backward();  aux = model.aux_loss();  aux.backward()

as a fixed sequence of hand-written CUDA launches over pre-allocated HBM buffers:

  * every conv / transposed conv runs the tcgen05 implicit-GEMM kernel (conv_tc.cu) forward, and the SAME
    kernel for its data gradient (dgrad of a stride-2 conv is a stride-2 transposed conv with the same weights
    and vice versa; stride-1 layers use the flipped pack);
  * weight gradients run on the tensor cores in wgrad_tc.cu (pixel reduction with MN-major operands straight
    from the NHWC activation / gradient buffers);
  * GDN is unfused in training (the pre-GDN activation and the norm are kept): x^2, a 1x1 tensor-core conv with
    gamma', x * rsqrt(norm); its backward is two element-wise passes around a 1x1 conv with gamma'^T and a 1x1
    weight gradient for gamma';
  * the entropy models produce their likelihoods AND the rate term's gradients in one pass (train_entropy.cu);
  * activations and gradients are NHWC bf16 (fp32 accumulation everywhere), latents / entropy parameters /
    images fp32; parameter gradients are fp32 views into ONE flat buffer (the all-reduce bucket of the
    data-parallel step, masic_b200/sharding.py).

Quantisation noise: the reference draws U(-.5,.5) inside the model (entropy_models.py:88-96, seven draws per
step); `step_grads(..., noise=...)` takes the seven tensors (oracle.train.NOISE_KEYS order / shapes) so parity
tests can feed both sides the same draw; with noise=None they are drawn on the device.

No CPU fallback: everything raises on non-CUDA tensors.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import _lib, ops
from . import train_ops as T
from ._lib import MasicError, check
from .convplan import (ACT_LEAKY, ACT_NONE, ACT_RELU, CONV, CONV_XFOLD8, DECONV_S2, DECONV_S2_SUBPIX, GDN_NONE,
                       MASK_A_5x5, ConvPlan, PackBatch, PackedConv, WgradPlan, gdn_prepare)

NOISE_KEYS = ("z1", "y1_ctx", "y1", "z2", "y2_ctx", "y1w", "y2")
XPAD = _lib.IMG_XPAD
IMG_CP = 8           # MASIC_CONV_XFOLD8 input pitch
BF = torch.bfloat16
F32 = torch.float32


def _flip_mask(mask: int, k: int) -> int:
    out = 0
    for ky in range(k):
        for kx in range(k):
            if mask & (1 << (ky * k + kx)):
                out |= 1 << ((k - 1 - ky) * k + (k - 1 - kx))
    return out


class _Layer:
    """One conv()/deconv() on the tensor cores: forward plan, data-gradient plan, weight-gradient plan."""

    def __init__(self, tr: "HSICTrainer", name: str, *, transposed: bool, k: int, stride: int, c_in: int, c_out: int,
                 x: torch.Tensor, out: torch.Tensor, in_coff: int = 0, out_coff: int = 0, act=ACT_NONE, n_tile: int = 0,
                 tap_mask: int = 0, gx: Optional[torch.Tensor] = None, gx_coff: int = 0, gout: Optional[torch.Tensor] = None,
                 weight: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                 dweight: Optional[torch.Tensor] = None, dbias: Optional[torch.Tensor] = None, accumulate: bool = False,
                 share: Optional["_Layer"] = None, wgrad_tap_mask: Optional[int] = None,
                 res0: Optional[torch.Tensor] = None, res1: Optional[torch.Tensor] = None,
                 act_out: Optional[torch.Tensor] = None, dg_n_tile: int = 0,
                 dg_res0: Optional[torch.Tensor] = None, dg_res0_coff: int = 0,
                 dg_res1: Optional[torch.Tensor] = None, dg_res1_coff: int = 0):
        """res0 / res1 / act_out: residual adds of the forward epilogue and the pre-residual activation store
        (ResidualBlock); dg_res0 / dg_res1: residual adds of the data gradient's epilogue (the skips' gradients)."""
        self.tr, self.name = tr, name
        self.transposed, self.k, self.stride, self.c_in, self.c_out = transposed, k, stride, c_in, c_out
        self.w = weight if weight is not None else tr.param(name + ".weight")
        self.b = bias if bias is not None else tr.param(name + ".bias")
        self.dw = dweight if dweight is not None else tr.grad(name + ".weight")
        self.db = dbias if dbias is not None else tr.grad(name + ".bias")
        self.x, self.out, self.in_coff, self.out_coff = x, out, in_coff, out_coff
        self.act, self.tap_mask = act, tap_mask
        self.gx, self.gx_coff, self.gout = gx, gx_coff, gout
        n_tile = n_tile or (128 if c_out % 192 else 192)
        if transposed and stride == 2:
            kind = DECONV_S2
        else:
            kind = CONV
        self.kind = kind
        # ---- forward
        if share is not None:
            self.pack = share.pack
        else:
            self.pack = PackedConv(kind=kind, ksize=k, c_in=c_in, c_out=c_out, n_tile=n_tile, weight=self.w,
                                   transposed=transposed, bias=self.b)
            tr.repack.append((self.pack, self.w, self.b))
        # CTA pairs where they measured faster in the inference engine: the 128 -> 128 5x5 stride-2 layers (and their
        # data gradients, which are the same operator transposed) and the wide 1x1 / 3x3 / masked layers
        pairs = (k == 5 and stride == 2 and c_in == 128 and c_out == 128 and not transposed) or (k == 1 and c_out >= 3000)
        self.fwd_plan = ConvPlan(packed=self.pack, stride=stride, tap_mask=tap_mask, x=x, in_coff=in_coff, out=out,
                                 out_coff=out_coff, act=act, cta_pairs=pairs, residual0=res0, residual1=res1,
                                 act_out=act_out)
        # ---- weight gradient: conv: LO = dL/dout, HI = input; deconv: LO = input, HI = dL/dout
        if gout is not None:
            if transposed:
                lo, c_lo, lo_coff, hi, c_hi, hi_coff = x, c_in, in_coff, gout, c_out, out_coff
            else:
                lo, c_lo, lo_coff, hi, c_hi, hi_coff = gout, c_out, out_coff, x, c_in, in_coff
            self.wg_plan = WgradPlan(ksize=k, stride=stride, lo=lo, c_lo=c_lo, lo_coff=lo_coff, hi=hi, c_hi=c_hi,
                                     hi_coff=hi_coff, dw=self.dw, accumulate=accumulate,
                                     tap_mask=tap_mask if wgrad_tap_mask is None else wgrad_tap_mask)
        # ---- data gradient: the transpose of the forward operator with the same weights
        self.dg_plan = None
        if gx is not None:
            if share is not None and share.dg_plan is not None:
                self.dpack = share.dpack
            else:
                if stride == 2:
                    dkind = CONV if transposed else DECONV_S2
                else:
                    dkind = CONV
                dn = dg_n_tile or (128 if c_in % 192 else 192)
                self.dpack = PackedConv(kind=dkind, ksize=k, c_in=c_out, c_out=c_in, n_tile=dn, weight=self.w,
                                        transposed=not transposed)
                tr.repack.append((self.dpack, self.w, None))
            self.dg_plan = ConvPlan(packed=self.dpack, stride=stride, tap_mask=_flip_mask(tap_mask, k) if tap_mask else 0,
                                    x=gout, in_coff=out_coff, out=gx, out_coff=gx_coff, residual0=dg_res0,
                                    res0_coff=dg_res0_coff, residual1=dg_res1, res1_coff=dg_res1_coff)

    def fwd(self):
        self.fwd_plan.launch()

    def bwd(self, skip_act: bool = False):
        """gout holds dL/d(activated output); turns it into dL/d(pre-activation) in place, then bias / weight /
        data gradients."""
        if not skip_act:
            acts = self.act if isinstance(self.act, (list, tuple)) else None
            if acts is None:
                T.act_bwd_bias(self.gout, self.out_coff, self.c_out, self.out if self.act != ACT_NONE else None,
                               self.out_coff, self.act, self.db)
            else:                                      # per n-tile activations (the fused 3-branch layer)
                nt = self.pack.n_tile
                i = 0
                while i < len(acts):
                    j = i
                    while j < len(acts) and acts[j] == acts[i]:
                        j += 1
                    c0, c1 = i * nt, min(j * nt, self.c_out)
                    T.act_bwd_bias(self.gout, self.out_coff + c0, c1 - c0, self.out if acts[i] != ACT_NONE else None,
                                   self.out_coff + c0, acts[i], self.db[c0:c1])
                    i = j
        self.tr.wg_async(self.wg_plan.launch)
        if self.dg_plan is not None:
            self.dg_plan.launch()


class _GDN:
    """GDN / IGDN over 128 channels, unfused (training): keeps x and the norm."""

    def __init__(self, tr: "HSICTrainer", name: str, inverse: bool, x: torch.Tensor, y: torch.Tensor,
                 gy: Optional[torch.Tensor], accumulate: bool = False, share: Optional["_GDN"] = None):
        self.tr, self.name, self.inverse, self.x, self.y, self.gy = tr, name, inverse, x, y, gy
        dev = x.device
        c = x.shape[-1]
        self.c = c
        self.beta, self.gamma = tr.param(name + ".beta"), tr.param(name + ".gamma")
        self.dbeta, self.dgamma = tr.grad(name + ".beta"), tr.grad(name + ".gamma")
        self.accumulate = accumulate
        self.sq = torch.zeros_like(x)
        self.norm = torch.zeros(*x.shape, dtype=F32, device=dev)
        if share is None:
            self.beta_p = torch.zeros(c, device=dev)
            self.gamma_p = torch.zeros(c, c, device=dev)
            self.gamma_pt = torch.zeros(c, c, device=dev)
            self.pk_n = PackedConv(ksize=1, c_in=c, c_out=c, n_tile=128, weight=self.gamma_p.view(c, c, 1, 1), bias=self.beta_p)
            self.pk_v = PackedConv(ksize=1, c_in=c, c_out=c, n_tile=128, weight=self.gamma_pt.view(c, c, 1, 1))
            tr.gdn_prep.append(self)
            self.dbeta_p = torch.zeros(c, device=dev)
            self.dgamma_p = torch.zeros(c, c, device=dev)
            tr.zero_each_step += [self.dbeta_p, self.dgamma_p]
            tr.gdn_finish.append(self)
            self._first = True
        else:
            self.beta_p, self.gamma_p, self.gamma_pt, self.pk_n, self.pk_v = (share.beta_p, share.gamma_p, share.gamma_pt,
                                                                              share.pk_n, share.pk_v)
            self.dbeta_p, self.dgamma_p = share.dbeta_p, share.dgamma_p
            self._first = False
        self.p_norm = ConvPlan(packed=self.pk_n, stride=1, x=self.sq, out=self.norm)
        if gy is not None:
            self.t = torch.zeros_like(x)
            self.v = torch.zeros(*x.shape, dtype=F32, device=dev)
            self.p_v = ConvPlan(packed=self.pk_v, stride=1, x=self.t, out=self.v)
            # dgamma' is zeroed every step and every pass through these parameters accumulates (encoder1 runs twice)
            self.wg = WgradPlan(ksize=1, stride=1, lo=self.t, c_lo=c, hi=self.sq, c_hi=c, dw=self.dgamma_p, accumulate=True)

    def prepare(self):
        """beta' / gamma' of this step (parametrizers.py:61-64) -> the two packed 1x1 weights."""
        lib = self.tr.lib
        check(lib.masic_gdn_prepare(self.beta.data_ptr(), self.gamma.data_ptr(), self.c, 1e-6, self.beta_p.data_ptr(),
                                    self.gamma_p.data_ptr(), None, 0, T._s()), "masic_gdn_prepare")
        self.gamma_pt.copy_(self.gamma_p.t())
        self.pk_n.repack(self.gamma_p.view(self.c, self.c, 1, 1), self.beta_p)
        self.pk_v.repack(self.gamma_pt.view(self.c, self.c, 1, 1))

    def fwd(self):
        T.gdn_square(self.x, self.sq)
        self.p_norm.launch()
        T.gdn_apply(self.x, self.norm, self.inverse, self.y)

    def bwd(self, dbias: Optional[torch.Tensor]):
        """gy (dL/dy) -> dL/dx in place (it is the pre-activation gradient of the conv that feeds this GDN);
        dbias += column sums (that conv's bias gradient)."""
        T.gdn_bwd_a(self.gy, self.x, self.norm, self.inverse, self.t, self.dbeta_p)
        self.p_v.launch()
        T.gdn_bwd_b(self.gy, self.x, self.v, dbias)
        self.tr.wg_async(self.wg.launch)

    def finish(self):
        T.reparam_bwd(self.dbeta_p, self.beta, 1e-6, self.dbeta)
        T.reparam_bwd(self.dgamma_p, self.gamma, 0.0, self.dgamma)


class _GDN3:
    """GDN(3) / IGDN(3) on NCHW fp32 images (pre_gdn, after_gdn)."""

    def __init__(self, tr, name, inverse):
        self.tr, self.inverse = tr, inverse
        self.beta, self.gamma = tr.param(name + ".beta"), tr.param(name + ".gamma")
        self.dbeta, self.dgamma = tr.grad(name + ".beta"), tr.grad(name + ".gamma")
        self.dbp = torch.zeros(3, device=tr.dev)
        self.dgp = torch.zeros(3, 3, device=tr.dev)
        tr.zero_each_step += [self.dbp, self.dgp]

    def fwd(self, x, y):
        ops.gdn_nchw_into(x, self.beta, self.gamma, y, inverse=self.inverse)

    def bwd(self, x, g, dx):
        T.gdn_small_bwd(x, g, self.beta, self.gamma, self.inverse, dx, self.dbp, self.dgp)
        T.reparam_bwd(self.dbp, self.beta, 1e-6, self.dbeta)
        T.reparam_bwd(self.dgp, self.gamma, 0.0, self.dgamma)


class TrainStep:
    """What every training step of this package shares: the flat gradient buffer, the weight re-packing, the
    forward / backward op lists with their lanes and the weight-gradient side stream, and the CUDA-graph replay.
    A subclass builds its ops in `_build()` and defines `_issue(refresh)`."""

    def _init_step(self, model, use_graph: bool):
        self.use_graph, self.graph, self._warm = use_graph, None, False
        self._params: Dict[str, torch.nn.Parameter] = dict(torch.nn.Module.named_parameters(model))
        for n, p in self._params.items():
            if not p.is_cuda or p.dtype != F32:
                raise MasicError(f"parameter {n} must be a CUDA fp32 tensor")
        total = sum(p.numel() for p in self._params.values())
        self.flat_grad = torch.zeros(total, device=self.dev)
        self._grads: Dict[str, torch.Tensor] = {}
        # Layout of the flat gradient buffer: the parameters in named_parameters() order, each gradient a view of its
        # slice, so that the data-parallel mean over the ranks is ONE all-reduce of the whole buffer (train_step).
        off = 0
        for n, p in self._params.items():
            self._grads[n] = self.flat_grad[off:off + p.numel()].view(p.shape)
            off += p.numel()
        self.repack: List[Tuple[PackedConv, torch.Tensor, Optional[torch.Tensor]]] = []
        self._pack_batch = None
        self.zero_each_step: List[torch.Tensor] = []
        self.fwd_ops: List[Tuple[str, Callable[[], None]]] = []
        self.bwd_ops: List[Tuple[str, Callable[[], None]]] = []
        self.pre_repack: List[Callable[[], None]] = []
        self.post_bwd: List[Callable[[], None]] = []

    def _make_streams(self):
        self._wg_stream = torch.cuda.Stream(device=self.dev)
        self._lane_streams: List[torch.cuda.Stream] = []

    # ------------------------------------------------------------------ helpers
    def param(self, name):
        return self._params[name]

    def grad(self, name):
        return self._grads[name]

    def _z(self, *shape, dtype=BF):
        return torch.zeros(*shape, dtype=dtype, device=self.dev)

    def F(self, name, fn):
        self.fwd_ops.append((name, fn))

    def Bk(self, name, fn):
        self.bwd_ops.append((name, fn))

    # Weight gradients are leaves of the backward pass: nothing downstream reads dW before the optimizer.  They are
    # issued on a SECOND stream (forked from the main stream at the point where their operands are final, joined once
    # before the reparametrisation / scatter ops that read the gradients), so the ~115 wgrad + reduce launches — most
    # of them at 1/8 and 1/16 resolution with fewer than 148 busy CTAs — overlap the data-gradient chain instead of
    # extending it.  All of them share ONE side stream: they also share one partial-sum workspace.  Every operand
    # buffer of the step is allocated once and never reused, so the fork event is the only ordering they need.
    def wg_async(self, fn):
        ev = torch.cuda.Event()
        ev.record()
        self._wg_stream.wait_event(ev)
        with torch.cuda.stream(self._wg_stream):
            fn()

    def wg_join(self):
        ev = torch.cuda.Event()
        ev.record(self._wg_stream)
        torch.cuda.current_stream().wait_event(ev)

    def _repack_weights(self):
        """Re-pack every weight the kernels read from the model's current fp32 parameters."""
        for f in self.pre_repack:
            f()
        if self._pack_batch is None:
            ok = all(w.dtype == F32 and w.is_contiguous() and (b is None or (b.dtype == F32 and b.is_contiguous()))
                     for _, w, b in self.repack)
            self._pack_batch = PackBatch(self.repack) if ok else False
        if self._pack_batch:
            self._pack_batch.launch()                    # every weight pack and bias copy in one launch
        else:
            for pk, w, b in self.repack:
                pk.repack(w, b)

    def _run(self, refresh: bool):
        """One step: replayed as a CUDA graph once warm (eager issue through ctypes is host-bound, ~20 us per
        launch), issued eagerly otherwise; then `.grad` of every parameter points at its flat-buffer view."""
        if self.use_graph and self._warm and refresh:
            if self.graph is None:
                torch.cuda.synchronize(self.dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._issue(True)
                self.graph = g
            self.graph.replay()
        else:
            self._issue(refresh)
            self._warm = True
        for n, p in self._params.items():
            p.grad = self._grads[n]

    def _run_lanes(self, ops, lanes):
        main = torch.cuda.current_stream()
        while len(self._lane_streams) < len(lanes):
            self._lane_streams.append(torch.cuda.Stream(device=self.dev))
        on_lane = frozenset().union(*[l[0] for l in lanes])

        def fork(i):                                 # the lane sees everything issued on the main stream so far
            ev = torch.cuda.Event()
            ev.record(main)
            side = self._lane_streams[i]
            side.wait_event(ev)
            with torch.cuda.stream(side):
                for name, fn in ops:
                    if name in lanes[i][0]:
                        fn()

        joined = set()
        for i, (_, fork_after, _) in enumerate(lanes):
            if fork_after is None:
                fork(i)
        for name, fn in ops:
            if name in on_lane:
                continue
            for i, (_, _, join_before) in enumerate(lanes):
                if name == join_before:
                    ev = torch.cuda.Event()
                    ev.record(self._lane_streams[i])
                    main.wait_event(ev)
                    joined.add(i)
            fn()
            for i, (_, fork_after, _) in enumerate(lanes):
                if name == fork_after:
                    fork(i)
        assert len(joined) == len(lanes), "a lane was never joined"

    def profile(self, iters: int = 3):
        """CUDA-event time of every forward / backward op group (after one warm step)."""
        res = []
        with torch.cuda.device(self.dev):
            for name, fn in [("F:" + n, f) for n, f in self.fwd_ops] + [("B:" + n, f) for n, f in self.bwd_ops]:
                ts = []
                for _ in range(iters):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); fn(); e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                res.append((name, sorted(ts)[len(ts) // 2]))
        return res


class HSICTrainer(TrainStep):
    def __init__(self, model, batch: int, height: int, width: int, device, lmbda: float = 0.01,
                 use_graph: bool = True, metric: str = "mse"):
        """metric: the distortion term of the loss, per view.  "mse" is the reference's
        lambda * 255^2 * (mse1 + mse2) + bpp; "ms-ssim" is CompressAI's RateDistortionLoss(metric="ms-ssim") on both
        views, lambda * ((1 - ms1) + (1 - ms2)) + bpp with ms_v = pytorch_msssim.ms_ssim(x_v_hat, x_v, data_range=1.0)
        (MS-SSIM lambdas are on a different scale from MSE ones)."""
        if metric not in ("mse", "ms-ssim"):
            raise ValueError(f"metric must be 'mse' or 'ms-ssim', got {metric!r}")
        if metric == "ms-ssim" and min(height, width) <= 160:
            raise ValueError(f"metric='ms-ssim' needs min(H, W) > 160 (5 MS-SSIM levels), got {height}x{width}")
        if height % 64 or width % 64:
            raise ValueError("HSIC needs H and W to be multiples of 64")
        self.metric = metric
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("HSICTrainer runs on a CUDA device only (no CPU fallback)")
        self.model, self.B, self.H, self.W, self.lmbda = model, batch, height, width, float(lmbda)
        self.N, self.M, self.K = model.N, model.M, model.K
        if (self.N, self.M, self.K) != (128, 192, 5):
            raise MasicError("the sm_100a kernels are specialised for HSIC(N=128, M=192, K=5)")
        self._init_step(model, use_graph)
        self.gdn_prep: List[_GDN] = []
        self.gdn_finish: List[_GDN] = []
        self.flops_fwd = 0.0
        with torch.cuda.device(self.dev):
            self._make_streams()
            self._build()

    # ------------------------------------------------------------------ sub-graphs
    def _encoder_pass(self, tag: str, enc: str, img_bf: torch.Tensor, img_nchw: torch.Tensor, accumulate: bool,
                      share: Optional[dict], need_dimg: bool):
        """g_a (MASIC.py:521-531): conv1..3 + GDN, conv4.  Returns dict with y (fp32 NHWC), gy (bf16 NHWC, to be
        filled by the caller before the pass's backward runs) and, if need_dimg, dimg (NCHW fp32 gradient)."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        d: dict = {"layers": [], "gdns": []}
        sizes = [(H // 2, W // 2), (H // 4, W // 4), (H // 8, W // 8)]
        prev, gprev = img_bf, None
        for i, (h, w) in enumerate(sizes, start=1):
            c = self._z(B, h, w, N)
            e = self._z(B, h, w, N)
            ge = self._z(B, h, w, N)               # dL/d(GDN out) -> dL/d(conv out) in place
            sh = share["layers"][i - 1] if share else None
            if i == 1:
                lay = _Conv1(self, f"{enc}.g_a_conv1", prev, img_nchw, c, ge, accumulate, sh, need_dimg)
            else:
                lay = _Layer(self, f"{enc}.g_a_conv{i}", transposed=False, k=5, stride=2, c_in=N, c_out=N, x=prev, out=c,
                             gx=gprev, gout=ge, accumulate=accumulate, share=sh)
            gd = _GDN(self, f"{enc}.g_a_gdn{i}", False, c, e, ge, accumulate, share["gdns"][i - 1] if share else None)
            d["layers"].append(lay); d["gdns"].append(gd)
            prev, gprev = e, ge
        y = self._z(B, H // 16, W // 16, M, dtype=F32)
        gy = self._z(B, H // 16, W // 16, M)
        l4 = _Layer(self, f"{enc}.g_a_conv4", transposed=False, k=5, stride=2, c_in=N, c_out=M, x=prev, out=y, gx=gprev,
                    gout=gy, accumulate=accumulate, share=share["layers"][3] if share else None, n_tile=192)
        d["layers"].append(l4)
        d["y"], d["gy"] = y, gy

        def fwd():
            for i in range(3):
                d["layers"][i].fwd()
                d["gdns"][i].fwd()
            l4.fwd()

        def bwd():
            l4.bwd()
            for i in (2, 1, 0):
                d["gdns"][i].bwd(d["layers"][i].db)
                d["layers"][i].bwd(skip_act=True)
        d["fwd"], d["bwd"] = fwd, bwd
        if need_dimg:
            d["dimg"] = d["layers"][0].dimg
        return d

    def _decoder_pass(self, tag: str, dec: str, y_bf: torch.Tensor, gy: torch.Tensor):
        """g_s (MASIC.py:544-554): deconv1..3 + IGDN, deconv4 in sub-pixel form.  Returns sp (fp32 NHWC
        [B,H/2,W/2,16], channel = phase*3+co) and the backward entry taking dL/d(image) NCHW fp32."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        sizes = [(H // 8, W // 8), (H // 4, W // 4), (H // 2, W // 2)]
        cins = [M, N, N]
        layers, gdns = [], []
        prev, gprev = y_bf, gy
        for i, (h, w) in enumerate(sizes, start=1):
            c = self._z(B, h, w, N)
            e = self._z(B, h, w, N)
            ge = self._z(B, h, w, N)
            lay = _Layer(self, f"{dec}.g_s_conv{i}", transposed=True, k=5, stride=2, c_in=cins[i - 1], c_out=N, x=prev, out=c,
                         gx=gprev, gout=ge, n_tile=128)
            gd = _GDN(self, f"{dec}.g_s_gdn{i}", True, c, e, ge)
            layers.append(lay); gdns.append(gd)
            prev, gprev = e, ge
        # deconv4: 128 -> 3, sub-pixel forward; backward = XFOLD4 conv of the padded gradient image + small wgrad
        w4, b4 = self.param(f"{dec}.g_s_conv4.weight"), self.param(f"{dec}.g_s_conv4.bias")
        dw4, db4 = self.grad(f"{dec}.g_s_conv4.weight"), self.grad(f"{dec}.g_s_conv4.bias")
        sp = self._z(B, H // 2, W // 2, 16, dtype=F32)
        p4 = PackedConv(kind=DECONV_S2_SUBPIX, ksize=5, c_in=N, c_out=3, n_tile=16, weight=w4, transposed=True, bias=b4)
        self.repack.append((p4, w4, b4))
        plan4 = ConvPlan(packed=p4, x=prev, out=sp)
        gimg_bf = self._z(B, H, W + XPAD, IMG_CP)
        d4 = PackedConv(kind=CONV_XFOLD8, ksize=5, c_in=64, c_out=N, n_tile=128, weight=w4)
        self.repack.append((d4, w4, None))
        dplan4 = ConvPlan(packed=d4, stride=2, x=gimg_bf, out=gprev)
        e3 = prev
        gimg16 = self._z(B, H, W, 16)                     # dense 16-pitch copy of dL/d(image) for the weight gradient
        dw16 = self._z(N, 16, 5, 5, dtype=F32)
        wg4 = WgradPlan(ksize=5, stride=2, lo=e3, c_lo=N, hi=gimg16, c_hi=16, dw=dw16)

        def fwd():
            for i in range(3):
                layers[i].fwd()
                gdns[i].fwd()
            plan4.launch()

        def bwd(gimg: torch.Tensor):
            """gimg: dL/d(deconv4 output image), NCHW fp32 (B,3,H,W)."""
            ops.nchw_to_nhwc_into(gimg, gimg_bf)
            T.colsum_nchw(gimg, db4)
            ops.nchw_to_nhwc_into(gimg, gimg16)
            self.wg_async(lambda: (wg4.launch(), dw4.add_(dw16[:, :3])))
            dplan4.launch()
            for i in (2, 1, 0):
                gdns[i].bwd(layers[i].db)
                layers[i].bwd(skip_act=True)
        return {"sp": sp, "fwd": fwd, "bwd": bwd}

    def _hyper(self, tag: str, idx: int, y_abs: torch.Tensor, g_yabs: torch.Tensor, p_out: torch.Tensor, p_coff: int,
               g_p: torch.Tensor, noise_key: str):
        """h_a -> EntropyBottleneck (train) -> h_s_up; params written to p_out[..., p_coff:p_coff+2M]."""
        B, H, W, N, M = self.B, self.H, self.W, self.N, self.M
        h16, w16 = H // 16, W // 16
        ha, hs, ebn = f"_h_a{idx}.encode_hyper", f"h_s{idx}_up", f"entropy_bottleneck{idx}"
        c1, g1 = self._z(B, h16, w16, N), self._z(B, h16, w16, N)
        c2, g2 = self._z(B, h16 // 2, w16 // 2, N), self._z(B, h16 // 2, w16 // 2, N)
        z = self._z(B, h16 // 4, w16 // 4, N, dtype=F32)
        gz = self._z(B, h16 // 4, w16 // 4, N)
        l1 = _Layer(self, f"{ha}.0", transposed=False, k=5, stride=1, c_in=M, c_out=N, x=y_abs, out=c1, act=ACT_RELU,
                    gx=g_yabs, gout=g1)
        l2 = _Layer(self, f"{ha}.2", transposed=False, k=5, stride=2, c_in=N, c_out=N, x=c1, out=c2, act=ACT_RELU, gx=g1,
                    gout=g2)
        l3 = _Layer(self, f"{ha}.4", transposed=False, k=5, stride=2, c_in=N, c_out=N, x=c2, out=z, gx=g2, gout=gz)
        mats = [self.param(f"{ebn}._matrices.{i}") for i in range(5)]
        bias = [self.param(f"{ebn}._biases.{i}") for i in range(5)]
        facs = [self.param(f"{ebn}._factors.{i}") for i in range(4)]
        hw64 = (h16 // 4) * (w16 // 4)
        z_hat = self._z(B, N, h16 // 4, w16 // 4, dtype=F32)
        z_lik = self._z(B, N, h16 // 4, w16 // 4, dtype=F32)
        zq, gzq = self._z(B, h16 // 4, w16 // 4, N), self._z(B, h16 // 4, w16 // 4, N)
        dz_lik = self._z(B, h16 // 4, w16 // 4, N, dtype=F32)
        dpar = self._z(N, 58, dtype=F32)
        d1, gd1 = self._z(B, h16 // 2, w16 // 2, M), self._z(B, h16 // 2, w16 // 2, M)
        d2, gd2 = self._z(B, h16, w16, 2 * M), self._z(B, h16, w16, 2 * M)          # 288 real channels
        s1 = _Layer(self, f"{hs}.0", transposed=True, k=5, stride=2, c_in=N, c_out=M, x=zq, out=d1, act=ACT_LEAKY, gx=gzq,
                    gout=gd1, n_tile=192)
        s2 = _Layer(self, f"{hs}.2", transposed=True, k=5, stride=2, c_in=M, c_out=M * 3 // 2, x=d1, out=d2, act=ACT_LEAKY,
                    gx=gd1, gout=gd2, n_tile=192)
        s3 = _Layer(self, f"{hs}.4", transposed=False, k=3, stride=1, c_in=M * 3 // 2, c_out=2 * M, x=d2, out=p_out,
                    out_coff=p_coff, gx=gd2, gout=g_p, n_tile=192)
        # s3's dgrad / wgrad read g_p at channel offset p_coff of the gradient buffer (same layout as p_out)
        offs = [0, 3, 12, 21, 30, 33, 36, 39, 42, 45, 46, 49, 52, 55, 58]
        targets = [self.grad(f"{ebn}._matrices.{i}") for i in range(5)] + [self.grad(f"{ebn}._biases.{i}") for i in range(5)] \
            + [self.grad(f"{ebn}._factors.{i}") for i in range(4)]
        scale = T.lik_grad_scale(B * H * W)

        def fwd():
            l1.fwd(); l2.fwd(); l3.fwd()
            T.eb_train(z, self.noise[noise_key], B, N, hw64, mats, bias, facs, scale, z_hat=z_hat, lik=z_lik, zq=zq,
                       dz=dz_lik, dparams=dpar)
            for i, t in enumerate(targets):
                t.copy_(dpar[:, offs[i]:offs[i + 1]].reshape(t.shape))
            s1.fwd(); s2.fwd(); s3.fwd()

        def bwd():
            s3.bwd(); s2.bwd(); s1.bwd()
            T.add_f32_bf16(dz_lik, gzq, gz)
            l3.bwd(); l2.bwd(); l1.bwd()
        return {"fwd": fwd, "bwd": bwd, "z_hat": z_hat, "z_lik": z_lik}

    def _gmm_net(self, tag: str, net: str, cin: int, first_is_deconv: bool, gmm_in: torch.Tensor, g_in: torch.Tensor):
        """Three 1x1 branches (MASIC.py:338-376 / :410-444), layer 0 fused into one wide GEMM."""
        B, H, W, M, K = self.B, self.H, self.W, self.M, self.K
        h16, w16 = H // 16, W // 16
        MK = M * K
        t = first_is_deconv
        br = ("gmm_sigma", "gmm_means", "gmm_weights")
        dev = self.dev
        # fused layer-0 weight/bias and their fused gradients (scattered to the three parameters after the step)
        w0 = torch.zeros((cin, 18 * M, 1, 1) if t else (18 * M, cin, 1, 1), device=dev)
        b0 = torch.zeros(18 * M, device=dev)
        dw0, db0 = torch.zeros_like(w0), torch.zeros_like(b0)
        self.zero_each_step += [db0]
        srcs_w = [self.param(f"{net}.{b}.0.weight") for b in br]
        srcs_b = [self.param(f"{net}.{b}.0.bias") for b in br]

        def gather():
            torch.cat(srcs_w, dim=1 if t else 0, out=w0)
            torch.cat(srcs_b, out=b0)
        self.pre_repack.append(gather)
        l0 = self._z(B, h16, w16, 18 * M)
        gl0 = self._z(B, h16, w16, 18 * M)
        L0 = _Layer(self, f"{net}.l0", transposed=t, k=1, stride=1, c_in=cin, c_out=18 * M, x=gmm_in, out=l0,
                    act=[ACT_RELU] * 6 + [ACT_LEAKY] * 12, n_tile=192, gx=g_in, gout=gl0, weight=w0, bias=b0, dweight=dw0,
                    dbias=db0)

        def scatter():
            for i, b in enumerate(br):
                sl = slice(6 * M * i, 6 * M * (i + 1))
                self.grad(f"{net}.{b}.0.weight").copy_(dw0[:, sl] if t else dw0[sl])
                self.grad(f"{net}.{b}.0.bias").copy_(db0[sl])
        self.post_bwd.append(scatter)
        l1, gl1 = self._z(B, h16, w16, 8 * M), self._z(B, h16, w16, 8 * M)
        l1w, gl1w = self._z(B, h16, w16, MK), self._z(B, h16, w16, MK)
        sig, mu, wl = (self._z(B, h16, w16, MK, dtype=F32) for _ in range(3))
        gsig, gmu, gwl = (self._z(B, h16, w16, MK) for _ in range(3))
        S1 = _Layer(self, f"{net}.gmm_sigma.2", transposed=t, k=1, stride=1, c_in=6 * M, c_out=4 * M, x=l0, in_coff=0, out=l1,
                    out_coff=0, act=ACT_RELU, gx=gl0, gx_coff=0, gout=gl1, n_tile=192)
        M1 = _Layer(self, f"{net}.gmm_means.2", transposed=t, k=1, stride=1, c_in=6 * M, c_out=4 * M, x=l0, in_coff=6 * M,
                    out=l1, out_coff=4 * M, act=ACT_LEAKY, gx=gl0, gx_coff=6 * M, gout=gl1, n_tile=192)
        W1 = _Layer(self, f"{net}.gmm_weights.2", transposed=t, k=1, stride=1, c_in=6 * M, c_out=MK, x=l0, in_coff=12 * M,
                    out=l1w, act=ACT_LEAKY, gx=gl0, gx_coff=12 * M, gout=gl1w, n_tile=192)
        # last layers: sigma's ReLU is applied by the forward epilogue and its derivative is folded into dsigma by
        # the likelihood kernel -> backward treats all three as linear
        S2 = _Layer(self, f"{net}.gmm_sigma.4", transposed=False, k=1, stride=1, c_in=4 * M, c_out=MK, x=l1, in_coff=0,
                    out=sig, act=ACT_RELU, gx=gl1, gx_coff=0, gout=gsig, n_tile=192)
        M2 = _Layer(self, f"{net}.gmm_means.4", transposed=False, k=1, stride=1, c_in=4 * M, c_out=MK, x=l1, in_coff=4 * M,
                    out=mu, gx=gl1, gx_coff=4 * M, gout=gmu, n_tile=192)
        W2 = _Layer(self, f"{net}.gmm_weights.4", transposed=False, k=1, stride=1, c_in=MK, c_out=MK, x=l1w, out=wl, gx=gl1w,
                    gout=gwl, n_tile=192)
        for L in (S2, M2, W2):
            L.act = ACT_NONE

        def fwd():
            for L in (L0, S1, M1, W1, S2, M2, W2):
                L.fwd()

        def bwd():
            for L in (W2, M2, S2, W1, M1, S1, L0):
                L.bwd()
        return {"fwd": fwd, "bwd": bwd, "sig": sig, "mu": mu, "wl": wl, "gsig": gsig, "gmu": gmu, "gwl": gwl}

    # ------------------------------------------------------------------ the plan
    def _build(self):
        B, H, W, N, M, K = self.B, self.H, self.W, self.N, self.M, self.K
        h16, w16 = H // 16, W // 16
        dev = self.dev
        self.noise = {k: self._z(B, (h16 // 4) if k.startswith("z") else h16, (w16 // 4) if k.startswith("z") else w16,
                                 N if k.startswith("z") else M, dtype=F32) for k in NOISE_KEYS}     # NHWC
        self.x1 = self._z(B, 3, H, W, dtype=F32)
        self.x2 = self._z(B, 3, H, W, dtype=F32)
        self.Hm = torch.eye(3, device=dev).repeat(B, 1, 1).contiguous()
        npx16 = B * h16 * w16
        scale = T.lik_grad_scale(B * H * W)
        mse_scale = self.lmbda * 255.0 ** 2 * 2.0 / (B * 3 * H * W)
        ms_scale = -self.lmbda / (B * 3)            # d(lambda (1 - mean over (B, 3) of MS-SSIM)) / d(sum of MS-SSIM)
        o = self.out = {"x1_hat": self._z(B, 3, H, W, dtype=F32), "x2_hat": self._z(B, 3, H, W, dtype=F32),
                        "lik_y1": self._z(B, h16, w16, M, dtype=F32), "lik_y2": self._z(B, h16, w16, M, dtype=F32),
                        "y1_hat": self._z(B, h16, w16, M, dtype=F32), "y2_hat": self._z(B, h16, w16, M, dtype=F32)}

        # ================= left view =================
        x1_bf = self._z(B, H, W + XPAD, IMG_CP)
        # encoder1 runs twice (MASIC.py:746,822): both passes ADD into the step's zeroed gradient buffer
        encA = self._encoder_pass("A", "encoder1", x1_bf, self.x1, accumulate=True, share=None, need_dimg=False)
        y1, gy1 = encA["y"], encA["gy"]
        y1_abs, g_y1abs = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        y1_ctx, g_y1ctx = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        y1_hat_bf, g_y1hat = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        dy1_lik = self._z(B, h16, w16, M, dtype=F32)
        gmm1_in, g_gmm1_in = self._z(B, h16, w16, 4 * M), self._z(B, h16, w16, 4 * M)
        hyp1 = self._hyper("L", 1, y1_abs, g_y1abs, gmm1_in, 0, g_gmm1_in, "z1")
        ctx1 = _Layer(self, "context_prediction1", transposed=False, k=5, stride=1, c_in=M, c_out=2 * M, x=y1_ctx,
                      out=gmm1_in, out_coff=2 * M, tap_mask=MASK_A_5x5, gx=g_y1ctx, gout=g_gmm1_in, n_tile=192, wgrad_tap_mask=0)
        net1 = self._gmm_net("L", "_h_s1_same_resolution", 4 * M, True, gmm1_in, g_gmm1_in)
        dec1 = self._decoder_pass("L", "decoder1", y1_hat_bf, g_y1hat)

        self.F("x1.pack", lambda: ops.nchw_to_nhwc_into(self.x1, x1_bf))
        self.F("L.encoder", encA["fwd"])
        self.F("L.latent_prep", lambda: T.latent_prep_train(y1, self.noise["y1_ctx"], y1_abs, y1_ctx))
        self.F("L.hyper", hyp1["fwd"])
        self.F("L.context", ctx1.fwd)
        self.F("L.gmm_net", net1["fwd"])
        self.F("L.likelihood", lambda: T.gmm_likelihood_train(
            y1, self.noise["y1"], net1["sig"], net1["mu"], net1["wl"], M, K, scale, lik=o["lik_y1"], y_hat_bf=y1_hat_bf,
            y_hat=o["y1_hat"], dy=dy1_lik, dsigma=net1["gsig"], dmu=net1["gmu"], dwl=net1["gwl"]))
        self.F("L.decoder", dec1["fwd"])
        self.F("L.x1_hat", lambda: ops.subpix_to_nchw_into(dec1["sp"], o["x1_hat"]))

        # ================= right view =================
        Tm = torch.empty(B, 3, 3, device=dev, dtype=torch.float64)
        self.F("warp.prepare", lambda: ops.warp_prepare_into(self.Hm, Tm, (H, W), (H, W)))
        mask_R = self._z(B, 1, H, W, dtype=F32)
        self.F("mask_R", lambda: ops.warp_perspective_into(None, Tm, (H, W), src_shape=mask_R.shape, dst=mask_R))
        # mask2weights (MASIC.py:472-506)
        mk = "mask2weights_unit.maskconv"
        kshape = [(1, H, W), (3, H // 2, W // 2), (6, H // 4, W // 4), (6, H // 8, W // 8), (3, h16, w16)]
        kb = [mask_R] + [self._z(B, *s, dtype=F32) for s in kshape[1:]]
        gk = [None] + [self._z(B, *s, dtype=F32) for s in kshape[1:]]
        mw = self._z(B, h16, w16, 3, dtype=F32)
        dmw = self._z(B, h16, w16, 3, dtype=F32)
        mk_w = [self.param(f"{mk}.{2 * i}.weight") for i in range(4)]
        mk_b = [self.param(f"{mk}.{2 * i}.bias") for i in range(4)]
        mk_dw = [self.grad(f"{mk}.{2 * i}.weight") for i in range(4)]
        mk_db = [self.grad(f"{mk}.{2 * i}.bias") for i in range(4)]

        def mask_fwd():
            for i in range(4):
                ops.conv_small_into(kb[i], None, mk_w[i], mk_b[i], ksize=3, stride=2, act=ACT_RELU if i < 3 else ACT_NONE,
                                    out=kb[i + 1])
            ops.softmax_channels_into(kb[4], out_nhwc=mw)
        self.F("mask2weights", mask_fwd)

        x1_warp = self._z(B, 3, H, W, dtype=F32)
        pc = self._z(B, 3, H, W, dtype=F32)           # pre_conv output (before pre_gdn)
        pg = self._z(B, 3, H, W, dtype=F32)           # pre_gdn output = encoder2's image
        d_pg = None
        x2in_bf = self._z(B, H, W + XPAD, IMG_CP)
        pre_w, pre_b = self.param("encoder2.pre_conv.weight"), self.param("encoder2.pre_conv.bias")
        pre_gdn = _GDN3(self, "encoder2.pre_gdn", False)
        self.F("R.warp(x1)", lambda: ops.warp_perspective_into(self.x1, Tm, (H, W), dst=x1_warp))
        self.F("R.pre_conv", lambda: ops.conv_small_into(x1_warp, self.x2, pre_w, pre_b, ksize=5, stride=1, out=pc))
        self.F("R.pre_gdn", lambda: pre_gdn.fwd(pc, pg))
        self.F("R.pack", lambda: ops.nchw_to_nhwc_into(pg, x2in_bf))
        encB = self._encoder_pass("B", "encoder2", x2in_bf, pg, accumulate=False, share=None, need_dimg=True)
        y2, gy2 = encB["y"], encB["gy"]
        y2_abs, g_y2abs = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        y2_ctx, g_y2ctx = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        y2_hat_bf, g_y2hat = self._z(B, h16, w16, M), self._z(B, h16, w16, M)
        dy2_lik = self._z(B, h16, w16, M, dtype=F32)
        P2, gP2 = self._z(B, h16, w16, 2 * M), self._z(B, h16, w16, 2 * M)
        C2, gC2 = self._z(B, h16, w16, 2 * M), self._z(B, h16, w16, 2 * M)
        hyp2 = self._hyper("R", 2, y2_abs, g_y2abs, P2, 0, gP2, "z2")
        ctx2 = _Layer(self, "context_prediction2", transposed=False, k=5, stride=1, c_in=M, c_out=2 * M, x=y2_ctx, out=C2,
                      tap_mask=MASK_A_5x5, gx=g_y2ctx, gout=gC2, n_tile=192, wgrad_tap_mask=0)
        self.F("R.encoder", encB["fwd"])
        self.F("R.latent_prep", lambda: T.latent_prep_train(y2, self.noise["y2_ctx"], y2_abs, y2_ctx))
        self.F("R.hyper", hyp2["fwd"])
        self.F("R.context", ctx2.fwd)

        # x1_hat warped once (MASIC.py:821 == :833), encoder1 again on it (:822)
        x1hw = self._z(B, 3, H, W, dtype=F32)
        x1hw_bf = self._z(B, H, W + XPAD, IMG_CP)
        self.F("R.warp(x1_hat)", lambda: ops.warp_perspective_into(o["x1_hat"], Tm, (H, W), dst=x1hw, dst16=x1hw_bf))
        encC = self._encoder_pass("C", "encoder1", x1hw_bf, x1hw, accumulate=True, share=encA, need_dimg=True)
        y1w, gy1w = encC["y"], encC["gy"]
        self.F("R.encoder1(x1_hat_warp)", encC["fwd"])
        gmm2_in, g_gmm2_in = self._z(B, h16, w16, 5 * M), self._z(B, h16, w16, 5 * M)
        self.F("R.mask_fuse", lambda: T.mask_fuse_fwd(P2, C2, y1w, self.noise["y1w"], mw, gmm2_in))
        net2 = self._gmm_net("R", "_h_s2_same_resolution", 5 * M, False, gmm2_in, g_gmm2_in)
        self.F("R.gmm_net", net2["fwd"])
        self.F("R.likelihood", lambda: T.gmm_likelihood_train(
            y2, self.noise["y2"], net2["sig"], net2["mu"], net2["wl"], M, K, scale, lik=o["lik_y2"], y_hat_bf=y2_hat_bf,
            y_hat=o["y2_hat"], dy=dy2_lik, dsigma=net2["gsig"], dmu=net2["gmu"], dwl=net2["gwl"]))
        dec2 = self._decoder_pass("R", "decoder2", y2_hat_bf, g_y2hat)
        core = self._z(B, 3, H, W, dtype=F32)          # decoder2 core output (before after_gdn)
        ag = self._z(B, 3, H, W, dtype=F32)            # after_gdn output
        after_gdn = _GDN3(self, "decoder2.after_gdn", True)
        aw, ab = self.param("decoder2.after_conv.weight"), self.param("decoder2.after_conv.bias")
        self.F("R.decoder", dec2["fwd"])
        self.F("R.core", lambda: ops.subpix_to_nchw_into(dec2["sp"], core))
        self.F("R.after_gdn", lambda: after_gdn.fwd(core, ag))
        self.F("R.after_conv", lambda: ops.conv_small_into(ag, x1hw, aw, ab, ksize=5, stride=1, transposed_s1=True,
                                                           out=o["x2_hat"]))
        o["z1_hat"], o["lik_z1"], o["z2_hat"], o["lik_z2"] = hyp1["z_hat"], hyp1["z_lik"], hyp2["z_hat"], hyp2["z_lik"]

        # ================= loss =================
        self.rd_out = self._z(8, dtype=F32)
        self.rd_scratch = ops.rd_metrics_scratch(dev)
        liks = [o["lik_y1"], o["lik_y2"], o["lik_z1"], o["lik_z2"]]
        if self.metric == "mse":
            self.F("loss", lambda: ops.rd_metrics_into(liks, o["x1_hat"], self.x1, o["x2_hat"], self.x2, self.lmbda,
                                                       self.rd_scratch, self.rd_out))
        else:
            # bpp and the MSEs stay as diagnostics; each view's MS-SSIM keeps its own scratch for its backward
            self.ms_out = self._z(2, B, 3, dtype=F32)
            self.ms_res = self._z(3, dtype=F32)                   # ms1, ms2, loss
            s1, self.ms_work = T.ms_ssim_buffers(B, 3, H, W, dev)  # one work: the backward calls run one by one
            self.ms_scratch = [s1, T.ms_ssim_buffers(B, 3, H, W, dev)[0]]

            def loss():
                ops.rd_metrics_into(liks, o["x1_hat"], self.x1, o["x2_hat"], self.x2, self.lmbda, self.rd_scratch,
                                    self.rd_out)
                T.ms_ssim_fwd(o["x1_hat"], self.x1, self.ms_scratch[0], self.ms_out[0])
                T.ms_ssim_fwd(o["x2_hat"], self.x2, self.ms_scratch[1], self.ms_out[1])
                torch.mean(self.ms_out, dim=(1, 2), out=self.ms_res[0:2])
                torch.add(self.rd_out[6:7], self.lmbda * (2.0 - self.ms_res[0:2].sum()), out=self.ms_res[2:3])
            self.F("loss", loss)
        # aux loss (entropy_models.py:345-348) of both bottlenecks
        self.aux_out = self._z(1, dtype=F32)
        self.zero_each_step += [self.aux_out]

        aux_targets = {idx: getattr(self.model, f"entropy_bottleneck{idx}").target.tolist() for idx in (1, 2)}

        def aux():
            for idx in (1, 2):
                ebn = f"entropy_bottleneck{idx}"
                mats = [self.param(f"{ebn}._matrices.{i}") for i in range(5)]
                bias = [self.param(f"{ebn}._biases.{i}") for i in range(5)]
                facs = [self.param(f"{ebn}._factors.{i}") for i in range(4)]
                tgt = aux_targets[idx]
                T.eb_aux_loss(self.param(f"{ebn}.quantiles"), N, mats, bias, facs, tgt, self.aux_out,
                              self.grad(f"{ebn}.quantiles"))
        self.F("aux_loss", aux)

        # ================= backward =================
        gx2 = self._z(B, 3, H, W, dtype=F32)
        d_ag = self._z(B, 3, H, W, dtype=F32)
        d_x1hw_a = self._z(B, 3, H, W, dtype=F32)
        d_core = self._z(B, 3, H, W, dtype=F32)
        adw, adb = self.grad("decoder2.after_conv.weight"), self.grad("decoder2.after_conv.bias")
        if self.metric == "mse":
            self.Bk("mse2", lambda: T.mse_grad(o["x2_hat"], self.x2, mse_scale, gx2))
        else:
            self.Bk("mse2", lambda: T.ms_ssim_grad(o["x2_hat"], self.x2, self.ms_scratch[1], ms_scale, gx2,
                                                   work=self.ms_work))
        self.Bk("after_conv", lambda: T.conv_small_bwd(ag, x1hw, aw, True, 3, 5, 1, gx2, din0=d_ag, din1=d_x1hw_a, dweight=adw,
                                                       dbias=adb))
        self.Bk("after_gdn", lambda: after_gdn.bwd(core, d_ag, d_core))
        self.Bk("R.decoder", lambda: dec2["bwd"](d_core))
        # g_y2hat now holds dL/dy2_hat from the decoder; GMM-net 2 backward from the likelihood gradients
        self.Bk("R.gmm_net", net2["bwd"])
        gY1W = gy1w       # dL/d(y1w): straight into encoder pass C's output gradient

        self.Bk("R.mask_fuse", lambda: T.mask_fuse_bwd(g_gmm2_in, P2, C2, y1w, self.noise["y1w"], mw, gP2, gC2, gY1W, dmw))

        def mask_bwd():
            T.softmax_channels_bwd(mw, dmw, B, 3, h16 * w16, gk[4])
            for i in (3, 2, 1, 0):
                T.conv_small_bwd(kb[i], None, mk_w[i], False, kshape[i + 1][0], 3, 2, gk[i + 1],
                                 act_out=kb[i + 1] if i < 3 else None, din0=gk[i] if i > 0 else None, dweight=mk_dw[i],
                                 dbias=mk_db[i])
        self.Bk("mask2weights", mask_bwd)
        self.Bk("R.encoder1(x1_hat_warp)", encC["bwd"])
        d_x1hw_b = self._z(B, 3, H, W, dtype=F32)
        self.Bk("C.dimg", lambda: ops.subpix_to_nchw_into(encC["dimg"], d_x1hw_b))
        d_x1hat_w = self._z(B, 3, H, W, dtype=F32)
        self.zero_each_step += [d_x1hat_w]
        self.Bk("warp_bwd", lambda: T.warp_bwd(d_x1hw_a, d_x1hw_b, Tm, d_x1hat_w))
        self.Bk("R.context", ctx2.bwd)
        self.Bk("R.hyper", hyp2["bwd"])
        self.Bk("R.latent_merge", lambda: T.latent_merge_bwd(y2, dy2_lik, g_y2hat, g_y2ctx, g_y2abs, gy2))
        self.Bk("R.encoder", encB["bwd"])
        d_pgt = self._z(B, 3, H, W, dtype=F32)
        d_pc = self._z(B, 3, H, W, dtype=F32)
        pdw, pdb = self.grad("encoder2.pre_conv.weight"), self.grad("encoder2.pre_conv.bias")
        self.Bk("B.dimg", lambda: ops.subpix_to_nchw_into(encB["dimg"], d_pgt))
        self.Bk("pre_gdn", lambda: pre_gdn.bwd(pc, d_pgt, d_pc))
        self.Bk("pre_conv", lambda: T.conv_small_bwd(x1_warp, self.x2, pre_w, False, 3, 5, 1, d_pc, dweight=pdw, dbias=pdb))
        # left view
        gx1 = self._z(B, 3, H, W, dtype=F32)
        if self.metric == "mse":
            self.Bk("mse1", lambda: T.mse_grad(o["x1_hat"], self.x1, mse_scale, gx1, addend=d_x1hat_w))
        else:
            self.Bk("mse1", lambda: T.ms_ssim_grad(o["x1_hat"], self.x1, self.ms_scratch[0], ms_scale, gx1,
                                                   addend=d_x1hat_w, work=self.ms_work))
        self.Bk("L.decoder", lambda: dec1["bwd"](gx1))
        self.Bk("L.gmm_net", net1["bwd"])
        self.Bk("L.context", ctx1.bwd)
        self.Bk("L.hyper", hyp1["bwd"])
        self.Bk("L.latent_merge", lambda: T.latent_merge_bwd(y1, dy1_lik, g_y1hat, g_y1ctx, g_y1abs, gy1))
        self.Bk("L.encoder", encA["bwd"])
        # the 2 x 15 reparam backwards of the fused-GDN layers as one launch
        self._reparam = T.ReparamBatch([j for g in self.gdn_finish for j in ((g.dbeta_p, g.beta, 1e-6, g.dbeta),
                                                                             (g.dgamma_p, g.gamma, 0.0, g.dgamma))])
        self.Bk("wgrad.join", self.wg_join)
        self.Bk("gdn.reparam", self._reparam.launch)
        self.Bk("scatter", lambda: [f() for f in self.post_bwd])
        # hyper-synthesis conv3x3 of the LEFT view writes / reads channel slice [0, 2M) of the 4M-wide gmm1_in; its
        # gradient arrives in g_gmm1_in[..., 0:2M] (written by net1's layer-0 dgrad) — same layout, nothing to do.

    # ------------------------------------------------------------------ running
    @torch.no_grad()
    def refresh_weights(self):
        """Re-pack every weight the kernels read from the model's current fp32 parameters (~110 weight packs and ~50
        bias copies in one launch) and prepare the GDN layers' effective parameters."""
        self._repack_weights()
        for g in self.gdn_prep:
            g.prepare()
        # MaskedConv2d side effect (layers.py:77) is applied through tap_mask; keep the parameter masked too
        with torch.no_grad():
            for cp in (self.model.context_prediction1, self.model.context_prediction2):
                cp.weight.data *= cp.mask

    @torch.no_grad()
    def step_grads(self, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor,
                   noise: Optional[Dict[str, torch.Tensor]] = None, refresh: bool = True,
                   read_back: bool = True) -> Optional[Dict[str, float]]:
        """One forward + backward.  Fills `.grad` of every model parameter (views of `flat_grad`): the main loss's
        gradient everywhere, the aux loss's gradient on the bottleneck quantiles (as the reference's two optimisers
        see them).  noise: NCHW fp32 tensors keyed by NOISE_KEYS, or None to draw U(-.5,.5) on the device."""
        with torch.cuda.device(self.dev):
            self._load_inputs(x1, x2, h_matrix, noise)
            # the ~700 launches of a step (zeroing, weight re-packing, forward, backward) replayed as ONE CUDA graph
            self._run(refresh)
            return self.read_losses() if read_back else None

    def _load_inputs(self, x1, x2, h_matrix, noise):
        self.x1.copy_(x1, non_blocking=True)
        self.x2.copy_(x2, non_blocking=True)
        self.Hm.copy_(h_matrix.reshape(self.B, 3, 3), non_blocking=True)
        for k in NOISE_KEYS:
            if noise is None:
                self.noise[k].uniform_(-0.5, 0.5)
            else:
                self.noise[k].copy_(noise[k].permute(0, 2, 3, 1))

    def read_losses(self) -> Dict[str, float]:
        """Loss terms of the last step (one device -> host read; synchronises with the step)."""
        if self.metric == "mse":
            r = torch.cat([self.rd_out, self.aux_out]).tolist()
            return {"loss": r[7], "bpp": r[6], "mse": r[4] + r[5], "aux": r[8]}
        r = torch.cat([self.rd_out, self.aux_out, self.ms_res]).tolist()
        return {"loss": r[11], "bpp": r[6], "mse": r[4] + r[5], "aux": r[8], "msssim1": r[9], "msssim2": r[10]}

    # Lanes, like the inference engine's: the right view's own encoder chain (homography products, mask weights,
    # pre_conv, encoder2, hyperprior 2, context 2) depends on nothing the left view computes, and its backward
    # (everything below R.mask_fuse that is not the second encoder1 pass) feeds nothing but weight gradients.  These ops
    # are issued on a second stream: forked from the main stream where the lane starts, joined where its results are
    # first read (forward: R.mask_fuse; backward: the final join).  Every buffer is allocated once per trainer and
    # written by one op only, so the two events per phase are the only ordering needed.
    # (op names of the lane, fork after this main-stream op (None = start of the phase), join before this main-stream op)
    FWD_LANES = ((frozenset(("warp.prepare", "mask_R", "mask2weights", "R.warp(x1)", "R.pre_conv", "R.pre_gdn", "R.pack",
                            "R.encoder", "R.latent_prep", "R.hyper", "R.context")),
                  None, "R.warp(x1_hat)"),)            # the main stream first reads the lane's prepared homography there
    BWD_LANES = ((frozenset(("mask2weights", "R.context", "R.hyper", "R.latent_merge", "R.encoder", "B.dimg", "pre_gdn",
                            "pre_conv")),
                  "R.mask_fuse", "wgrad.join"),)       # inputs complete after R.mask_fuse; only weight gradients come out
    # (measured and dropped: a third lane for L.gmm_net / L.context / L.hyper from the start of the backward pass,
    # joined before L.latent_merge: 8.37 vs 8.28 ms — the lanes already keep the SMs busy)

    def _issue(self, refresh: bool):
        self.flat_grad.zero_()
        for t in self.zero_each_step:
            t.zero_()
        if refresh:
            self.refresh_weights()
        self._run_lanes(self.fwd_ops, self.FWD_LANES)
        self._run_lanes(self.bwd_ops, self.BWD_LANES)

    def train_step(self, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor, optimizer, aux_optimizer,
                   noise: Optional[Dict[str, torch.Tensor]] = None, group=None,
                   clip_max_norm: Optional[float] = None) -> Dict[str, float]:
        """One iteration of newtrain_codec_real.py:105-146 on this rank's batch: forward + backward, the data-parallel
        gradient all-reduce (mean over ranks: the loss normalises by the LOCAL batch, :76), then both optimisers.
        `optimizer` holds model.parameters() (everything but the bottlenecks), `aux_optimizer` model.aux_parameters()
        (MASIC.py:77-94).  The gradients live in ONE flat fp32 buffer, so the all-reduce is a single NCCL call over
        NVLink/NVSwitch (35 M floats = 140 MB); nothing else is communicated."""
        # the loss scalars are read back AFTER the optimisers are enqueued: the host does not wait for the step's graph
        # before it launches the all-reduce and the two Adam steps
        from .sharding import all_reduce_mean_
        self.step_grads(x1, x2, h_matrix, noise=noise, read_back=False)
        all_reduce_mean_(self.flat_grad, group=group)                 # one collective; no-op on a single rank
        if clip_max_norm is not None and clip_max_norm > 0:
            # torch.nn.utils.clip_grad_norm_(model.parameters(), clip_max_norm) of CompressAI's training loops, on the
            # flat buffer: the main parameters' gradients (everything but the two bottlenecks, MASIC.py:77-94)
            if getattr(self, "_main_grads", None) is None:
                aux_ids = {id(p) for p in self.model.aux_parameters()}
                self._main_grads = [self._grads[n] for n, p in self._params.items() if id(p) not in aux_ids]
            total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(g) for g in self._main_grads]))
            coef = torch.clamp(clip_max_norm / (total + 1e-6), max=1.0)
            torch._foreach_mul_(self._main_grads, coef)
        optimizer.step()
        aux_optimizer.step()
        return self.read_losses()


class _Conv1:
    """g_a_conv1 (Conv2d 3 -> 128, k5 s2): XFOLD4 tensor-core forward on the padded bf16 image, CUDA-core weight
    gradient (3-channel side), sub-pixel transposed conv for the data gradient (encoder2 / second encoder1 pass)."""

    def __init__(self, tr: HSICTrainer, name: str, img_bf: torch.Tensor, img_nchw: torch.Tensor, out: torch.Tensor,
                 gout: torch.Tensor, accumulate: bool, share: Optional["_Conv1"], need_dimg: bool):
        self.tr = tr
        self.w, self.b = tr.param(name + ".weight"), tr.param(name + ".bias")
        self.dw, self.db = tr.grad(name + ".weight"), tr.grad(name + ".bias")
        self.img_nchw, self.gout = img_nchw, gout
        N = out.shape[-1]
        if share is None:
            self.pack = PackedConv(kind=CONV_XFOLD8, ksize=5, c_in=64, c_out=N, n_tile=128, weight=self.w, bias=self.b)
            tr.repack.append((self.pack, self.w, self.b))
            self.dpack = PackedConv(kind=DECONV_S2_SUBPIX, ksize=5, c_in=N, c_out=3, n_tile=16, weight=self.w, transposed=True)
            tr.repack.append((self.dpack, self.w, None))
        else:
            self.pack, self.dpack = share.pack, share.dpack
        self.fwd_plan = ConvPlan(packed=self.pack, stride=2, x=img_bf, out=out)
        self.dimg = None
        self.dg_plan = None
        if need_dimg:
            B, h, w, _ = out.shape
            self.dimg = torch.zeros(B, h, w, 16, dtype=F32, device=out.device)
            self.dg_plan = ConvPlan(packed=self.dpack, x=gout, out=self.dimg)
        # weight gradient on the tensor cores: the image as a dense 16-channel-pitch NHWC operand (3 real channels),
        # dW lands in a (128, 16, 5, 5) scratch whose first 3 input channels are added to the parameter's gradient
        # (the CUDA-core masic_wgrad_small took ~0.5 ms per launch at 512x896 b2: a fifth of the whole step)
        Bn, _, Hh, Ww = img_nchw.shape
        self.img16 = torch.zeros(Bn, Hh, Ww, 16, dtype=torch.bfloat16, device=out.device)
        self.dw16 = torch.zeros(N, 16, 5, 5, dtype=F32, device=out.device)
        self.wg_plan = WgradPlan(ksize=5, stride=2, lo=gout, c_lo=N, hi=self.img16, c_hi=16, dw=self.dw16)

    def fwd(self):
        self.fwd_plan.launch()

    def bwd(self, skip_act: bool = True):
        ops.nchw_to_nhwc_into(self.img_nchw, self.img16)
        self.tr.wg_async(lambda: (self.wg_plan.launch(), self.dw.add_(self.dw16[:, :3])))
        if self.dg_plan is not None:
            self.dg_plan.launch()
