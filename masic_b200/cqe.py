"""Independent_EN — MASIC's cross quality enhancement (CQE) network on the B200-native kernels.

Mirror of `Independent_EN` (coremasic/mywork/MASIC.py:1436-1501) with its helper blocks
`Enhancement_Block` (:149-164), `mask2weights_EN` (:1411-1434) and compressai's `ResidualBlock`
(layers/layers.py:160-190): same constructor, same 86 `state_dict` entries created in the same order with the
same initialisers (`torch.manual_seed(s); Independent_EN()` draws the reference's weights), same
`forward(x1_hat, x2_hat, h_matrix) -> {"x1_hat", "x2_hat"}`.

`forward` hands the state_dict to a `CQEEngine` compiled for (batch, H, W): per view 21 tensor-core conv launches
(3x3, stride 1, 16/32/64/96 channels, NHWC bf16) with LeakyReLU and both kinds of skip connection fused into the
conv epilogue, plus the memory-bound glue of csrc/cqe.cu and csrc/image.cu (warps, masks, mask weights, blends).
The whole sequence replays as one CUDA graph.  No CPU path.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import MasicError
from .convplan import ACT_LEAKY, ACT_NONE, ACT_RELU, CONV, ConvPlan, PackedConv
from .engine import HSICEngine
from .layers import ResidualBlock, conv, conv3x3

F16 = _lib.FMT_F16              # inference runs on fp16 operands / activations (csrc/cvt16.cuh)


class Enhancement_Block(nn.Module):
    """MASIC.py:149-164 — three ResidualBlocks and a skip over all of them."""

    def __init__(self, shape: int):
        super().__init__()
        self.RB1 = ResidualBlock(shape, shape)
        self.RB2 = ResidualBlock(shape, shape)
        self.RB3 = ResidualBlock(shape, shape)

    def forward(self, x):
        return self.RB3(self.RB2(self.RB1(x))) + x


class mask2weights_EN(nn.Module):
    """MASIC.py:1411-1434 — 4x conv3 s1 (ReLU between) on a 1-channel mask, softmax over the Kw outputs."""

    def __init__(self, Kw: int = 2):
        super().__init__()
        self.maskconv = nn.Sequential(
            conv(in_channels=1, out_channels=Kw, kernel_size=3, stride=1), nn.ReLU(inplace=True),
            conv(in_channels=Kw, out_channels=Kw * 2, kernel_size=3, stride=1), nn.ReLU(inplace=True),
            conv(in_channels=Kw * 2, out_channels=Kw * 2, kernel_size=3, stride=1), nn.ReLU(inplace=True),
            conv(in_channels=Kw * 2, out_channels=Kw, kernel_size=3, stride=1))

    def forward(self, allconcat):
        x = allconcat
        for i in (0, 2, 4, 6):
            m = self.maskconv[i]
            x = ops.conv_small(x, None, m.weight, m.bias, ksize=3, stride=1, act=ACT_RELU if i < 6 else ACT_NONE)
        self.maskconvout = x
        self.weights = ops.softmax_channels(x)
        return self.weights


class Independent_EN(nn.Module):
    def __init__(self, use_cuda_graph: bool = True):
        super().__init__()
        self.EBl1 = Enhancement_Block(shape=32)          # MASIC.py:1440-1449 (creation order kept)
        self.EBl2 = Enhancement_Block(shape=64)
        self.EBl3 = Enhancement_Block(shape=96)
        self.EBr1 = Enhancement_Block(shape=32)
        self.EBr2 = Enhancement_Block(shape=64)
        self.EBr3 = Enhancement_Block(shape=96)
        self.conv0 = conv3x3(3, 32)
        self.conv1 = conv3x3(6, 32)
        self.conv2 = conv3x3(96, 3)
        self.mask2weights_unit = mask2weights_EN()
        self._use_graph = use_cuda_graph
        self._engines: Dict[Tuple, "CQEEngine"] = {}

    def invalidate_engines(self):
        self._engines.clear()

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        res = super().load_state_dict(state_dict, strict=strict, **kw)
        self.invalidate_engines()
        return res

    def engine_for(self, batch: int, height: int, width: int, device) -> "CQEEngine":
        key = (batch, height, width, str(device), tuple(p._version for p in self.parameters()))
        eng = self._engines.get(key)
        if eng is None:
            self._engines.clear()
            eng = CQEEngine(self.state_dict(), batch, height, width, device, use_graph=self._use_graph)
            self._engines[key] = eng
        return eng

    def trainer(self, batch: int, height: int, width: int, device, lmbda: float = 0.01):
        """The CUDA training step of stage two (the codec frozen): `CQETrainer.step_grads` fills `.grad` of every
        parameter from lmbda * 255^2 * (mse1 + mse2) of the enhanced pair against the originals, `train_step` also
        all-reduces the gradients and steps the optimiser.  H and W must be multiples of 64."""
        from .cqe_trainer import CQETrainer
        return CQETrainer(self, batch, height, width, device, lmbda=lmbda)

    def forward(self, x1_hat: torch.Tensor, x2_hat: torch.Tensor, h_matrix: torch.Tensor, clone: bool = True):
        if not x1_hat.is_cuda:
            raise MasicError("Independent_EN.forward needs CUDA tensors: masic_b200 has no CPU fallback")
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()) and self.training:
            raise MasicError("Independent_EN.forward runs inference only on the CUDA engine (call .eval() / "
                             "torch.no_grad()); the training step (forward, loss, backward) runs as fused CUDA kernels "
                             "through model.trainer(batch, H, W, device, lmbda).train_step(...)")
        b, _, h, w = x1_hat.shape
        o = self.engine_for(b, h, w, x1_hat.device).run(x1_hat, x2_hat, h_matrix)
        c = (lambda t: t.clone()) if clone else (lambda t: t)
        return {"x1_hat": c(o["x1_hat"]), "x2_hat": c(o["x2_hat"])}


class CQEEngine(HSICEngine):
    """Execution plan of Independent_EN.forward for a fixed (batch, H, W): static buffers, conv plans, one graph.

    `inputs` (optional): caller-owned device tensors (x1_hat, x2_hat, h_matrix), two (B,3,H,W) fp32 and one (B,3,3)
    fp32, that the engine reads in place (PairStream binds a slot's codec outputs and homography).  The graph is
    captured against their pointers and `run()` copies nothing; by default the engine owns those buffers and `run`
    copies its arguments into them."""

    def __init__(self, sd: Dict[str, torch.Tensor], batch: int, height: int, width: int,
                 device: torch.device | str = "cuda:0", use_graph: bool = True,
                 inputs: Optional[Sequence[torch.Tensor]] = None):
        if height < 2 or width < 2:
            raise ValueError("Independent_EN needs H, W >= 2 (kornia's normalised grid divides by size-1)")
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("CQEEngine runs on a CUDA device only (no CPU fallback)")
        self.B, self.H, self.W = batch, height, width
        self.bound = inputs is not None
        if self.bound:
            if len(inputs) != 3:
                raise MasicError("CQEEngine inputs: (x1_hat, x2_hat, h_matrix)")
            shapes = ((batch, 3, height, width), (batch, 3, height, width), (batch, 3, 3))
            for t, shape in zip(inputs, shapes):
                if not (t.device == self.dev and t.dtype == torch.float32 and t.is_contiguous()
                        and tuple(t.shape) == shape):
                    raise MasicError(f"CQEEngine inputs must be contiguous float32 tensors of shapes {shapes} on "
                                     f"{self.dev}; got {tuple(t.shape)} {t.dtype} on {t.device}")
            self.x1, self.x2, self.Hm = inputs
        self.sd = {k: v.detach().to(self.dev) for k, v in sd.items()}
        self.steps, self.sched, self._lane = [], [], 0
        self.plans, self.buf, self.packs, self._keep = {}, {}, {}, []
        self.graph, self.use_graph = None, use_graph
        with torch.cuda.device(self.dev):
            self._build()

    # ------------------------------------------------------------------ helpers
    def _pack3(self, prefix: str, c_in: int, c_out: int, n_tile: int, real_cin: int | None = None) -> PackedConv:
        w = self._w(prefix + ".weight")
        if real_cin is not None:                 # 3 / 6 image channels inside a 16-channel pitch
            wp = torch.zeros(w.shape[0], c_in, 3, 3, device=self.dev)
            wp[:, :real_cin] = w
            w = wp
        return PackedConv(kind=CONV, ksize=3, c_in=c_in, c_out=c_out, n_tile=n_tile, weight=w,
                          bias=self._w(prefix + ".bias"), f16=F16)

    def _c3(self, name, packed, x, out, *, out_coff=0, act=ACT_NONE, res0=None, res1=None, res1_coff=0):
        plan = ConvPlan(packed=packed, stride=1, x=x, out=out, out_coff=out_coff, act=act, residual0=res0,
                        residual1=res1, res1_coff=res1_coff)
        self.plans[name] = plan
        self._add(name, plan.launch)

    def _enh_block(self, tag: str, prefix: str, ch: int, x, out, out_coff: int = 0):
        """Enhancement_Block (MASIC.py:156-164): RB1, RB2, RB3 then + x.  Each ResidualBlock (layers.py:175-190) is two
        launches: conv1 + LeakyReLU, then conv2 + LeakyReLU + identity (the block-level identity rides on RB3's)."""
        B, H, W = self.B, self.H, self.W
        t = self._buf(B, H, W, ch)
        cur = x
        for i in (1, 2, 3):
            p1 = self._pack3(f"{prefix}.RB{i}.conv1", ch, ch, ch)
            p2 = self._pack3(f"{prefix}.RB{i}.conv2", ch, ch, ch)
            self._c3(f"{tag}.RB{i}.conv1", p1, cur, t, act=ACT_LEAKY)
            if i < 3:
                nxt = self._buf(B, H, W, ch)
                self._c3(f"{tag}.RB{i}.conv2+skip", p2, t, nxt, act=ACT_LEAKY, res0=cur)
                cur = nxt
            else:
                self._c3(f"{tag}.RB3.conv2+skips", p2, t, out, out_coff=out_coff, act=ACT_LEAKY, res0=cur, res1=x)

    # ------------------------------------------------------------------ the plan
    def _build(self):
        B, H, W = self.B, self.H, self.W
        f32 = torch.float32
        if not self.bound:
            self.x1 = self._buf(B, 3, H, W, dtype=f32)       # inputs: the codec's reconstructions
            self.x2 = self._buf(B, 3, H, W, dtype=f32)
            self.Hm = torch.eye(3, device=self.dev).repeat(B, 1, 1).contiguous()
        o = self.out = {"x1_hat": self._buf(B, 3, H, W, dtype=f32), "x2_hat": self._buf(B, 3, H, W, dtype=f32)}
        T = torch.empty(B, 3, 3, device=self.dev, dtype=torch.float64)
        Tinv = torch.empty(B, 3, 3, device=self.dev, dtype=torch.float64)
        self._add("warp.prepare", lambda: (ops.warp_prepare_into(self.Hm, T, (H, W), (H, W)),
                                           ops.warp_prepare_into(self.Hm, Tinv, (H, W), (H, W), invert=True)))

        def warp(tag, src, Tm, dst):
            self._add(tag, lambda: ops.warp_perspective_into(src, Tm, (H, W), src_shape=dst.shape, dst=dst))

        # masks (MASIC.py:1458 -> :627-649) and the per-pixel blend weights (:1459-1460)
        mask_r = self._buf(B, 1, H, W, dtype=f32)
        mask_l = self._buf(B, 1, H, W, dtype=f32)
        warp("mask_R=warp(ones)", None, T, mask_r)
        warp("mask_L=warp(mask_R,Hinv)", mask_r, Tinv, mask_l)
        mk = "mask2weights_unit.maskconv"
        wts = {}
        mws = [self._w(f"{mk}.{i}.weight") for i in (0, 2, 4, 6)]
        mbs = [self._w(f"{mk}.{i}.bias") for i in (0, 2, 4, 6)]
        for side, m in (("R", mask_r), ("L", mask_l)):
            wt = self._buf(B, 2, H, W, dtype=f32)
            self._add(f"mask2weights_{side}(4 convs+softmax)",
                      lambda m=m, wt=wt: ops.cqe_mask_weights_into(m, mws, mbs, wt))
            wts[side] = wt
        self.buf["w_R"], self.buf["w_L"] = wts["R"], wts["L"]

        # warped images (:1461, :1464) and bf16 NHWC copies of the inputs
        x1w = self._buf(B, 3, H, W, dtype=f32)
        x2w = self._buf(B, 3, H, W, dtype=f32)
        warp("warp(x1_hat,H)", self.x1, T, x1w)
        warp("warp(x2_hat,Hinv)", self.x2, Tinv, x2w)
        p_conv0 = self._pack3("conv0", 16, 32, 32, real_cin=3)
        p_conv1 = self._pack3("conv1", 16, 32, 32, real_cin=6)
        p_conv2 = self._pack3("conv2", 96, 3, 16)
        views = (("L", "EBl", self.x1, x2w, wts["L"], Tinv, "x1_hat"),
                 ("R", "EBr", self.x2, x1w, wts["R"], T, "x2_hat"))
        e1 = {}
        cat96 = {}
        for v, eb, x_self, x_other_w, wt, _, _ in views:
            xbf = self._buf(B, H, W, 16)
            self._add(f"{v}.pack_nhwc", lambda x_self=x_self, xbf=xbf: ops.nchw_to_nhwc_into(x_self, xbf))
            cat96[v] = self._buf(B, H, W, 96)                 # [EB2 output | conv0(x)]  (:1486-1487)
            self._c3(f"{v}.conv0", p_conv0, xbf, cat96[v], out_coff=64)                      # :1467-1468
            blend = self._buf(B, H, W, 16)
            self._add(f"{v}.blend_images", lambda a=x_other_w, b=x_self, wt=wt, blend=blend:
                      ops.cqe_blend_images_into(a, b, wt, blend))                           # :1470-1471
            f1 = self._buf(B, H, W, 32)
            self._c3(f"{v}.conv1", p_conv1, blend, f1)                                       # :1473-1474
            e1[v] = self._buf(B, H, W, 32)
            self._enh_block(f"{v}.EB1", f"{eb}1", 32, f1, e1[v])                             # :1476-1477
        for v, eb, x_self, _, wt, Tm, okey in views:
            other = "R" if v == "L" else "L"
            fused = self._buf(B, H, W, 64)
            self._add(f"{v}.feature_fuse", lambda s=e1[v], ot=e1[other], wt=wt, Tm=Tm, fused=fused:
                      ops.cqe_feature_fuse_into(s, ot, wt, Tm, fused))                      # :1479-1482
            self._enh_block(f"{v}.EB2", f"{eb}2", 64, fused, cat96[v], out_coff=0)           # :1483-1484
            e3 = self._buf(B, H, W, 96)
            self._enh_block(f"{v}.EB3", f"{eb}3", 96, cat96[v], e3)                          # :1488-1489
            c2 = self._buf(B, H, W, 16, dtype=f32)
            self._c3(f"{v}.conv2", p_conv2, e3, c2)                                          # :1491-1492
            self._add(f"{v}.residual_image", lambda c2=c2, x_self=x_self, dst=o[okey]:
                      ops.cqe_residual_image_into(c2, x_self, dst))                         # :1495-1496
        self.flops = sum(p.flops for p in self.plans.values())

    def run(self, x1: Optional[torch.Tensor] = None, x2: Optional[torch.Tensor] = None,
            h_matrix: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        if self.bound and not (x1 is None and x2 is None and h_matrix is None):
            raise MasicError("this CQEEngine reads the tensors it was built with in place: call run() without inputs")
        return super().run(x1, x2, h_matrix)
