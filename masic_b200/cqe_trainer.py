"""CQETrainer — the training step of the cross quality enhancement network `Independent_EN` on the B200 kernels.

MASIC trains in two stages: the codec HSIC first (trainer.HSICTrainer), then, with the codec frozen, the enhancement
network on the codec's decoded pairs (the reference's coremasic/mywork/newtrain_cqe_real.py, which is not part of
this repository; SURVEY §2 records that it freezes HSIC).  One step restates

    out  = Independent_EN(x1_hat, x2_hat, h)                                   MASIC.py:1436-1501
    loss = lmbda * 255^2 * (mse(out["x1_hat"], x1) + mse(out["x2_hat"], x2))
    loss.backward()

The loss is the distortion term of RateDistortionLoss (newtrain_codec_real.py:66-87).  With the codec frozen its
rate term is a constant with no gradient, so it is left out; no reference checkout was available to check the stage-two
script's loss against, so this is the RateDistortionLoss restatement of masic_rd_metrics with no likelihoods.

Format as in HSICTrainer: activations and gradients NHWC bf16, fp32 accumulation, images NCHW fp32, parameter
gradients fp32 views into one flat buffer in named_parameters() order.  Every buffer is allocated once and written by
one op.  The 42 3x3 convolutions run on the tensor cores (forward, data gradient with the flipped pack, weight gradient
on the side stream).  conv0 (3 input channels), conv1 (6) and conv2 (3 outputs) run in 16-channel pitches on
zero-padded copies of their weights; their weight gradients land in padded staging tensors that are sliced into the
parameters' gradients after the step.  conv0 needs no data gradient (its input is the decoded image); conv1's data
gradient feeds only the mask-weight gradient of the image blend.

ResidualBlock (layers.py:175-190), r = LReLU(conv2(LReLU(conv1(x)))) + x, Enhancement_Block adding + x0 on RB3:
the forward epilogue of conv2 also stores LReLU(conv2(.)) before the adds (masic_conv_plan_set_act_out), since the
LeakyReLU derivative needs that sign and act + x rounded to bf16 loses it where |act| << |x|.  Backward: the
LeakyReLU derivative of conv2 is applied out of place (dL/dr is still read by the skip), and the skip gradients are
added in the epilogue of conv1's data gradient (RB1's also adds the outer skip's).

No CPU fallback: everything raises on non-CUDA tensors.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import _lib, ops
from . import train_ops as T
from ._lib import MasicError
from .convplan import ACT_LEAKY, ACT_NONE, ACT_RELU
from .trainer import BF, F32, TrainStep, _Layer

MASK_CH = ((1, 2), (2, 4), (4, 4), (4, 2))      # mask2weights_EN.maskconv (in, out) of layers 0, 2, 4, 6 (Kw = 2)


class CQETrainer(TrainStep):
    def __init__(self, model, batch: int, height: int, width: int, device, lmbda: float = 0.01,
                 use_graph: bool = True):
        if height <= 0 or width <= 0 or height % 64 or width % 64:
            raise ValueError("Independent_EN training needs H and W to be multiples of 64 (the codec's output sizes)")
        if batch <= 0:
            raise ValueError("batch must be positive")
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("CQETrainer runs on a CUDA device only (no CPU fallback)")
        self.model, self.B, self.H, self.W, self.lmbda = model, batch, height, width, float(lmbda)
        self._init_step(model, use_graph)
        self.layers: List[_Layer] = []
        with torch.cuda.device(self.dev):
            self._make_streams()
            self._build()

    # ------------------------------------------------------------------ pieces
    def _padded(self, name: str, shape, sl):
        """fp32 copy of parameter `name` zero-padded to `shape` (refreshed before every re-pack) and a staging tensor
        of the same shape for its weight gradient (sliced into the parameter's gradient after the step)."""
        src = self.param(name)
        wp = torch.zeros(*shape, device=self.dev)
        stage = torch.zeros(*shape, device=self.dev)
        self.pre_repack.append(lambda: wp[sl].copy_(src))
        self.zero_each_step.append(stage)
        dst = self.grad(name)
        self.post_bwd.append(lambda: dst.copy_(stage[sl]))
        return wp, stage

    def _conv3(self, name, **kw) -> _Layer:
        lay = _Layer(self, name, transposed=False, k=3, stride=1, **kw)
        self.layers.append(lay)
        return lay

    def _enh_block(self, prefix: str, ch: int, x, gx, out, gout):
        """Enhancement_Block (MASIC.py:149-164) over `ch` channels: x -> out (both at channel 0 of their buffers),
        gout = dL/d(out) -> gx = dL/dx.  Returns (fwd, bwd)."""
        B, H, W = self.B, self.H, self.W
        rbs = []
        xin, gin = x, gx
        for i in (1, 2, 3):
            a, ga = self._z(B, H, W, ch), self._z(B, H, W, ch)         # LReLU(conv1(.)) and its gradient
            z, gs = self._z(B, H, W, ch), self._z(B, H, W, ch)         # LReLU(conv2(.)) before the adds, its gradient
            o, go = (out, gout) if i == 3 else (self._z(B, H, W, ch), self._z(B, H, W, ch))
            c1 = self._conv3(f"{prefix}.RB{i}.conv1", c_in=ch, c_out=ch, x=xin, out=a, act=ACT_LEAKY, n_tile=ch,
                             gx=gin, gout=ga, dg_n_tile=ch, dg_res0=go, dg_res1=gout if i == 1 else None)
            c2 = self._conv3(f"{prefix}.RB{i}.conv2", c_in=ch, c_out=ch, x=a, out=o, act=ACT_LEAKY, n_tile=ch,
                             gx=ga, gout=gs, dg_n_tile=ch, res0=xin, res1=x if i == 3 else None, act_out=z)
            rbs.append((c1, c2, z, gs, go))
            xin, gin = o, go

        def fwd():
            for c1, c2, _, _, _ in rbs:
                c1.fwd()
                c2.fwd()

        def bwd():
            for c1, c2, z, gs, go in reversed(rbs):
                T.act_bwd_bias_out(go, 0, ch, z, 0, ACT_LEAKY, gs, 0, c2.db)
                c2.bwd(skip_act=True)
                c1.bwd()
        return fwd, bwd

    # ------------------------------------------------------------------ the plan
    def _build(self):
        B, H, W = self.B, self.H, self.W
        dev, hw = self.dev, H * W
        self.x1_hat, self.x2_hat = self._z(B, 3, H, W, dtype=F32), self._z(B, 3, H, W, dtype=F32)
        self.x1, self.x2 = self._z(B, 3, H, W, dtype=F32), self._z(B, 3, H, W, dtype=F32)
        self.Hm = torch.eye(3, device=dev).repeat(B, 1, 1).contiguous()
        o = self.out = {"x1_hat": self._z(B, 3, H, W, dtype=F32), "x2_hat": self._z(B, 3, H, W, dtype=F32)}
        Tm = torch.empty(B, 3, 3, device=dev, dtype=torch.float64)
        Tinv = torch.empty(B, 3, 3, device=dev, dtype=torch.float64)
        self.F("warp.prepare", lambda: (ops.warp_prepare_into(self.Hm, Tm, (H, W), (H, W)),
                                        ops.warp_prepare_into(self.Hm, Tinv, (H, W), (H, W), invert=True)))

        def warp(src, Tw, dst):
            ops.warp_perspective_into(src, Tw, (H, W), src_shape=dst.shape, dst=dst)

        # masks (MASIC.py:1458 -> :627-649) and mask2weights_EN (:1459-1460, :1411-1434), layer by layer so that the
        # backward has the intermediates; weights as NCHW (blends) and NHWC (softmax backward)
        mask_r, mask_l = self._z(B, 1, H, W, dtype=F32), self._z(B, 1, H, W, dtype=F32)
        self.F("masks", lambda: (warp(None, Tm, mask_r), warp(mask_r, Tinv, mask_l)))
        mk = "mask2weights_unit.maskconv"
        mk_w = [self.param(f"{mk}.{2 * i}.weight") for i in range(4)]
        mk_b = [self.param(f"{mk}.{2 * i}.bias") for i in range(4)]
        mk_dw = [self.grad(f"{mk}.{2 * i}.weight") for i in range(4)]
        mk_db = [self.grad(f"{mk}.{2 * i}.bias") for i in range(4)]
        side = {}
        for v, m in (("R", mask_r), ("L", mask_l)):
            kb = [m] + [self._z(B, co, H, W, dtype=F32) for _, co in MASK_CH]
            gk = [None] + [self._z(B, co, H, W, dtype=F32) for _, co in MASK_CH]
            wt, wt_nhwc, dwt = self._z(B, 2, H, W, dtype=F32), self._z(B, H, W, 2, dtype=F32), self._z(B, H, W, 2, dtype=F32)
            side[v] = {"kb": kb, "gk": gk, "wt": wt, "wt_nhwc": wt_nhwc, "dwt": dwt}

            def mask_fwd(kb=kb, wt=wt, wt_nhwc=wt_nhwc):
                for i in range(4):
                    ops.conv_small_into(kb[i], None, mk_w[i], mk_b[i], ksize=3, stride=1,
                                        act=ACT_RELU if i < 3 else ACT_NONE, out=kb[i + 1])
                ops.softmax_channels_into(kb[4], wt, wt_nhwc)
            self.F(f"{v}.mask2weights", mask_fwd)

        # padded copies of the small-channel layers (16-channel pitches, as CQEEngine._pack3)
        wp0, st0 = self._padded("conv0.weight", (32, 16, 3, 3), (slice(None), slice(0, 3)))
        wp1, st1 = self._padded("conv1.weight", (32, 16, 3, 3), (slice(None), slice(0, 6)))
        wp2, st2 = self._padded("conv2.weight", (16, 96, 3, 3), (slice(0, 3),))
        bp2 = torch.zeros(16, device=dev)
        b2 = self.param("conv2.bias")
        self.pre_repack.append(lambda: bp2[:3].copy_(b2))
        db2 = self.grad("conv2.bias")

        x_other_w = {"L": self._z(B, 3, H, W, dtype=F32), "R": self._z(B, 3, H, W, dtype=F32)}
        self.F("warp(x2_hat,Hinv)", lambda: warp(self.x2_hat, Tinv, x_other_w["L"]))                 # :1464
        self.F("warp(x1_hat,H)", lambda: warp(self.x1_hat, Tm, x_other_w["R"]))                      # :1461
        views = {"L": ("EBl", self.x1_hat, self.x1, Tinv, "x1_hat"), "R": ("EBr", self.x2_hat, self.x2, Tm, "x2_hat")}
        d: Dict[str, dict] = {}
        first: Dict[str, _Layer] = {}
        for v, (eb, xs, _, _, _) in views.items():
            e = d[v] = {}
            xbf = self._z(B, H, W, 16)
            e["cat96"], e["gcat96"] = self._z(B, H, W, 96), self._z(B, H, W, 96)            # [EB2 out | conv0(x)]
            e["conv0"] = self._conv3("conv0", c_in=16, c_out=32, x=xbf, out=e["cat96"], out_coff=64, n_tile=32,
                                     gout=e["gcat96"], weight=wp0, dweight=st0, accumulate=True, share=first.get("conv0"))
            blend, e["gblend"] = self._z(B, H, W, 16), self._z(B, H, W, 16, dtype=F32)
            f1, gf1 = self._z(B, H, W, 32), self._z(B, H, W, 32)
            e["conv1"] = self._conv3("conv1", c_in=16, c_out=32, x=blend, out=f1, n_tile=32, gx=e["gblend"], gout=gf1,
                                     weight=wp1, dweight=st1, accumulate=True, share=first.get("conv1"), dg_n_tile=16)
            first.setdefault("conv0", e["conv0"]); first.setdefault("conv1", e["conv1"])
            e["e1"], e["ge1"] = self._z(B, H, W, 32), self._z(B, H, W, 32)
            e["eb1"] = self._enh_block(f"{eb}1", 32, f1, gf1, e["e1"], e["ge1"])
            e["xbf"], e["blend"] = xbf, blend

            def front(xs=xs, xbf=xbf, blend=blend, e=e, v=v):
                ops.nchw_to_nhwc_into(xs, xbf)
                e["conv0"].fwd()                                                                     # :1467-1468
                ops.cqe_blend_images_into(x_other_w[v], xs, side[v]["wt"], blend)                    # :1470-1471
                e["conv1"].fwd()                                                                     # :1473-1474
                e["eb1"][0]()                                                                        # :1476-1477
            self.F(f"{v}.front", front)
        for v, (eb, xs, _, Tv, okey) in views.items():
            e, other = d[v], d["R" if v == "L" else "L"]
            e["fused"], e["gfused"] = self._z(B, H, W, 64), self._z(B, H, W, 64)
            e["eb2"] = self._enh_block(f"{eb}2", 64, e["fused"], e["gfused"], e["cat96"], e["gcat96"])
            e3, ge3 = self._z(B, H, W, 96), self._z(B, H, W, 96)
            e["eb3"] = self._enh_block(f"{eb}3", 96, e["cat96"], e["gcat96"], e3, ge3)
            e["c2"], e["gc2"] = self._z(B, H, W, 16, dtype=F32), self._z(B, H, W, 16)
            e["conv2"] = self._conv3("conv2", c_in=96, c_out=16, x=e3, out=e["c2"], n_tile=16, gx=ge3, gout=e["gc2"],
                                     weight=wp2, bias=bp2, dweight=st2, dbias=db2, accumulate=True,
                                     share=first.get("conv2"), dg_n_tile=96)
            first.setdefault("conv2", e["conv2"])

            def back(e=e, other=other, v=v, Tv=Tv, xs=xs, okey=okey):
                ops.cqe_feature_fuse_into(e["e1"], other["e1"], side[v]["wt"], Tv, e["fused"])        # :1479-1482
                e["eb2"][0]()                                                                        # :1483-1487
                e["eb3"][0]()                                                                        # :1488-1489
                e["conv2"].fwd()                                                                     # :1491-1492
                ops.cqe_residual_image_into(e["c2"], xs, o[okey])                                    # :1495-1496
            self.F(f"{v}.back", back)

        # ================= loss: lambda * 255^2 * (mse1 + mse2), masic_rd_metrics without likelihoods
        self.rd_out = self._z(8, dtype=F32)
        self.rd_scratch = ops.rd_metrics_scratch(dev)
        self.F("loss", lambda: ops.rd_metrics_into([None] * 4, o["x1_hat"], self.x1, o["x2_hat"], self.x2, self.lmbda,
                                                   self.rd_scratch, self.rd_out))

        # ================= backward
        mse_scale = self.lmbda * 255.0 ** 2 * 2.0 / (B * 3 * H * W)
        for v, (_, _, target, _, okey) in views.items():
            e = d[v]
            gimg = self._z(B, 3, H, W, dtype=F32)

            def tail_bwd(e=e, gimg=gimg, target=target, okey=okey):
                T.mse_grad(o[okey], target, mse_scale, gimg)
                ops.nchw_to_nhwc_into(gimg, e["gc2"])
                T.colsum_nchw(gimg, db2)
                e["conv2"].bwd(skip_act=True)
                e["eb3"][1]()
                e["conv0"].bwd()
                e["eb2"][1]()
            self.Bk(f"{v}.back", tail_bwd)
        # the fuse backward crosses the views: L's fused map warps EB1(R) by H^-1, R's warps EB1(L) by H
        for v in ("L", "R"):
            d[v]["d_self"], d[v]["acc"] = self._z(B, H, W, 32), self._z(B, H, W, 32, dtype=F32)
            self.zero_each_step.append(d[v]["acc"])

        def fuse_bwd():
            for v, (_, _, _, Tv, _) in views.items():
                e, other = d[v], d["R" if v == "L" else "L"]
                T.cqe_feature_fuse_bwd(e["gfused"], e["e1"], other["e1"], side[v]["wt"], Tv, e["d_self"], other["acc"],
                                       side[v]["dwt"])
            for v in ("L", "R"):
                T.add_f32_bf16(d[v]["acc"], d[v]["d_self"], d[v]["ge1"])
        self.Bk("feature_fuse", fuse_bwd)
        for v in ("L", "R"):
            e = d[v]

            def front_bwd(e=e, v=v):
                e["eb1"][1]()
                e["conv1"].bwd()
                T.cqe_blend_images_bwd(e["gblend"], x_other_w[v], views[v][1], side[v]["dwt"])
                sd = side[v]
                T.softmax_channels_bwd(sd["wt_nhwc"], sd["dwt"], B, 2, hw, sd["gk"][4])
                for i in (3, 2, 1, 0):
                    T.conv_small_bwd(sd["kb"][i], None, mk_w[i], False, MASK_CH[i][1], 3, 1, sd["gk"][i + 1],
                                     act_out=sd["kb"][i + 1] if i < 3 else None, din0=sd["gk"][i] if i > 0 else None,
                                     dweight=mk_dw[i], dbias=mk_db[i])
            self.Bk(f"{v}.front", front_bwd)
        self.Bk("wgrad.join", self.wg_join)
        self.Bk("scatter", lambda: [f() for f in self.post_bwd])

    # ------------------------------------------------------------------ running
    def flops(self) -> float:
        """FLOPs of one step's tensor-core convolutions as planned (forward + data + weight gradients; the padded
        layers counted at their 16-channel pitch)."""
        tot = 0.0
        for lay in self.layers:
            tot += lay.fwd_plan.flops + lay.wg_plan.flops + (lay.dg_plan.flops if lay.dg_plan is not None else 0.0)
        return tot

    @torch.no_grad()
    def refresh_weights(self):
        """Re-pack every weight the kernels read from the model's current fp32 parameters."""
        self._repack_weights()

    def _issue(self, refresh: bool):
        self.flat_grad.zero_()
        for t in self.zero_each_step:
            t.zero_()
        if refresh:
            self.refresh_weights()
        for _, fn in self.fwd_ops:
            fn()
        for _, fn in self.bwd_ops:
            fn()

    def _load_inputs(self, x1_hat, x2_hat, h_matrix, x1, x2):
        shape = (self.B, 3, self.H, self.W)
        for name, t in (("x1_hat", x1_hat), ("x2_hat", x2_hat), ("x1", x1), ("x2", x2)):
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise MasicError(f"CQETrainer: {name} must be a CUDA tensor (no CPU fallback)")
            if tuple(t.shape) != shape:
                raise ValueError(f"CQETrainer: {name} has shape {tuple(t.shape)}, the trainer was built for {shape}")
        if not isinstance(h_matrix, torch.Tensor) or not h_matrix.is_cuda:
            raise MasicError("CQETrainer: h_matrix must be a CUDA tensor (no CPU fallback)")
        if h_matrix.numel() != self.B * 9:
            raise ValueError(f"CQETrainer: h_matrix must hold {self.B} 3x3 matrices")
        self.x1_hat.copy_(x1_hat, non_blocking=True)
        self.x2_hat.copy_(x2_hat, non_blocking=True)
        self.x1.copy_(x1, non_blocking=True)
        self.x2.copy_(x2, non_blocking=True)
        self.Hm.copy_(h_matrix.reshape(self.B, 3, 3), non_blocking=True)

    @torch.no_grad()
    def step_grads(self, x1_hat: torch.Tensor, x2_hat: torch.Tensor, h_matrix: torch.Tensor, x1: torch.Tensor,
                   x2: torch.Tensor, refresh: bool = True, read_back: bool = True) -> Optional[Dict[str, float]]:
        """One forward + loss + backward.  x*_hat: the codec's decoded pair, x1 / x2: the originals, all (B,3,H,W)
        fp32 CUDA tensors.  Fills `.grad` of every parameter (views of `flat_grad`, named_parameters() order).
        refresh=False skips re-packing the weights (they have not changed since the last step)."""
        with torch.cuda.device(self.dev):
            self._load_inputs(x1_hat, x2_hat, h_matrix, x1, x2)
            self._run(refresh)
            return self.read_losses() if read_back else None

    def read_losses(self) -> Dict[str, float]:
        """Loss terms of the last step (one device -> host read; synchronises with the step)."""
        r = self.rd_out.tolist()
        return {"loss": r[7], "mse1": r[4], "mse2": r[5], "mse": r[4] + r[5]}

    def train_step(self, x1_hat: torch.Tensor, x2_hat: torch.Tensor, h_matrix: torch.Tensor, x1: torch.Tensor,
                   x2: torch.Tensor, optimizer, group=None, clip_max_norm: Optional[float] = None) -> Dict[str, float]:
        """step_grads on this rank's batch, the data-parallel gradient mean (one all-reduce of the flat buffer,
        1.56 M floats), the optional clip_grad_norm_ over all parameters, optimizer.step().  The loss is read back
        after the optimiser is enqueued, so the host does not wait for the step first."""
        from .sharding import all_reduce_mean_
        self.step_grads(x1_hat, x2_hat, h_matrix, x1, x2, read_back=False)
        all_reduce_mean_(self.flat_grad, group=group)
        if clip_max_norm is not None and clip_max_norm > 0:
            total = torch.linalg.vector_norm(self.flat_grad)
            self.flat_grad.mul_(torch.clamp(clip_max_norm / (total + 1e-6), max=1.0))
        optimizer.step()
        return self.read_losses()
