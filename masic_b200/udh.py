"""The udh homography front-end on the B200 kernels (SURVEY §8(f)#4): two 128x128 grey patches -> h_matrix.

Same surface as the reference's `Net` (coremasic/mywork/model.py:73-111; wrapped by `HomographyModel`,
test2_real.py:42-47): constructor `Net(batch_norm=False, patch_size=128)`, `forward(a, b) -> delta (B,4,2)`,
`get_h(a, b, corners)`, and a state_dict with the reference's keys (`cnn.{0..3}.layers.{0,2}.{weight,bias}`,
`fc.{2,5}.{weight,bias}`), so udh checkpoints load unchanged.  `homography(a, b, corners, img_hw)` is the whole
chain the eval script runs per pair (test2_real.py:201-211): net -> 4-point DLT -> inverse -> h_adjust, as one CUDA
graph that never leaves the device — `HSIC.pair_stream().submit_patches(...)` feeds it straight into the codec.

Execution (UDHEngine): the eight 3x3 convolutions (+ReLU) are conv_tc plans on NHWC bf16 (2 -> 16-channel padded
input), max-pools one small kernel each, the two Linear layers a weight-streaming GEMV kernel (64 MB of bf16 weights
per call: HBM-bound), the DLT / inverse / h_adjust one thread per pair in fp64.  Inference only; CPU tensors raise.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import MasicError, check
from .convplan import ACT_RELU, ConvPlan, PackedConv

F16 = _lib.FMT_F16              # inference runs on fp16 operands / activations (csrc/cvt16.cuh)
ACT = _lib.act_dtype(F16)

PIC_SIZE = 256          # test2_real.py:40 — the views are resized to 256x256 before the 128x128 patches are cut


class _Block(nn.Module):
    """model.py:52-69 (batch_norm=False)."""

    def __init__(self, cin: int, cout: int, pool: bool = True):
        super().__init__()
        layers = [nn.Conv2d(cin, cout, kernel_size=3, padding=1), nn.ReLU(),
                  nn.Conv2d(cout, cout, kernel_size=3, padding=1), nn.ReLU()]
        if pool:
            layers.append(nn.MaxPool2d(2, 2))
        self.layers = nn.Sequential(*layers)


class _Flatten(nn.Module):
    def forward(self, x):
        return x.view(x.size(0), -1)


class Net(nn.Module):
    def __init__(self, batch_norm: bool = False, patch_size: int = 128):
        super().__init__()
        if batch_norm:
            raise MasicError("udh Net: batch_norm=True is not on the sm_100a path (the reference uses False)")
        self.patch_size = int(patch_size)
        self.cnn = nn.Sequential(_Block(2, 64), _Block(64, 64), _Block(64, 128), _Block(128, 128, pool=False))
        self.fc = nn.Sequential(_Flatten(), nn.Dropout(p=0.5), nn.Linear(128 * (patch_size // 8) ** 2, 1024), nn.ReLU(),
                                nn.Dropout(p=0.5), nn.Linear(1024, 4 * 2))
        self._engines: Dict[Tuple, "UDHEngine"] = {}

    def _engine(self, batch: int, device) -> "UDHEngine":
        key = (batch, str(device), tuple(p._version for p in self.parameters()))
        eng = self._engines.get(key)
        if eng is None:
            self._engines.clear()
            eng = self._engines[key] = UDHEngine(self.state_dict(), batch, device, self.patch_size)
        return eng

    def forward(self, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
        """model.py:95-100: delta (B, 4, 2)."""
        if self.training:
            raise MasicError("udh Net: the sm_100a path implements inference (eval mode)")
        if not a.is_cuda:
            raise MasicError("udh Net needs CUDA tensors: masic_b200 has no CPU fallback")
        return self._engine(a.shape[0], a.device).run(a, b)["delta"].clone()

    def get_h(self, a, b, corners):
        """model.py:102-111: inverse(get_perspective_transform(corners, corners + delta)) — corners as given, no
        h_adjust (the kernel's scaling by img/pic = 1 is exact)."""
        eng = self._engine(a.shape[0], a.device)
        return eng.run(a, b, corners, img_hw=(PIC_SIZE, PIC_SIZE), shift_corners=False)["h"].clone()

    def homography(self, a, b, corners, img_hw: Tuple[int, int]) -> torch.Tensor:
        """test2_real.py:201-211: the h_matrix HSIC.forward takes for views of size img_hw."""
        eng = self._engine(a.shape[0], a.device)
        return eng.run(a, b, corners, img_hw=img_hw)["h"].clone()


class UDHEngine:
    def __init__(self, sd: Dict[str, torch.Tensor], batch: int, device, patch_size: int = 128, use_graph: bool = True):
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise MasicError("UDHEngine runs on a CUDA device only (no CPU fallback)")
        if batch > 8:
            raise MasicError("UDHEngine: batch <= 8 (the FC kernel keeps one accumulator per batch row)")
        if patch_size % 16:
            raise MasicError("udh Net: patch_size must be a multiple of 16")
        self.B, self.P = batch, patch_size
        self.use_graph, self.graph, self._graph_key = use_graph, None, None
        sd = {k: v.detach().to(self.dev).float().contiguous() for k, v in sd.items()}
        with torch.cuda.device(self.dev):
            self._build(sd)

    def _build(self, sd):
        B, P, dev = self.B, self.P, self.dev
        bf = ACT
        self.corners = torch.zeros(B, 4, 2, device=dev)
        self.x_in = torch.zeros(B, P, P, 16, dtype=bf, device=dev)         # channels 0/1 = the two patches, rest zero
        self.steps = []
        self.plans = []
        chans = [(2, 64), (64, 64), (64, 128), (128, 128)]
        x, size = self.x_in, P
        for bi, (cin, cout) in enumerate(chans):
            for li, (ci, co) in enumerate(((cin, cout), (cout, cout))):
                w = sd[f"cnn.{bi}.layers.{2 * li}.weight"]
                if ci < 16:                                                   # 2 -> 16 input channels (zero weights)
                    wp = torch.zeros(co, 16, 3, 3, device=dev)
                    wp[:, :ci] = w
                    w, ci = wp, 16
                y = torch.zeros(B, size, size, co, dtype=bf, device=dev)
                pk = PackedConv(ksize=3, c_in=ci, c_out=co, n_tile=64 if co == 64 else 128, weight=w,
                                bias=sd[f"cnn.{bi}.layers.{2 * li}.bias"], f16=F16)
                plan = ConvPlan(packed=pk, stride=1, x=x, out=y, act=ACT_RELU)
                self.plans.append(plan)
                self.steps.append((f"cnn.{bi}.conv{li}", plan.launch))
                x = y
            if bi < 3:                                                        # MaxPool2d(2, 2)
                y = torch.zeros(B, size // 2, size // 2, cout, dtype=bf, device=dev)
                self.steps.append((f"cnn.{bi}.maxpool", (lambda xi=x, yo=y, s=size, c=cout: check(
                    self.lib.masic_maxpool2_nhwc_bf16(xi.data_ptr(), B, s, s, c, yo.data_ptr(), F16, self._s()),
                    "masic_maxpool2_nhwc_bf16"))))
                x, size = y, size // 2
        self.feat = x                                                         # (B, P/8, P/8, 128) bf16
        hw, k1 = size * size, 128 * size * size
        w1, w2 = sd["fc.2.weight"], sd["fc.5.weight"]
        if tuple(w1.shape) != (1024, k1):
            raise MasicError(f"udh Net: fc.2.weight is {tuple(w1.shape)}, expected (1024, {k1})")
        self.w1 = torch.empty(1024, k1, dtype=bf, device=dev)
        check(self.lib.masic_fc_pack_weights(w1.data_ptr(), 1024, 128, hw, self.w1.data_ptr(), F16, self._s()), "masic_fc_pack_weights")
        self.w2 = w2.to(bf).contiguous()
        self.b1, self.b2 = sd["fc.2.bias"], sd["fc.5.bias"]
        self.h1 = torch.zeros(B, 1024, dtype=bf, device=dev)
        self.delta = torch.zeros(B, 4, 2, device=dev)
        self.h = torch.zeros(B, 3, 3, device=dev)
        self.flops = sum(p.flops for p in self.plans) + 2.0 * B * (1024 * k1 + 8 * 1024)
        self.weight_bytes = 2.0 * (1024 * k1 + 8 * 1024)

    def _s(self):
        return torch.cuda.current_stream().cuda_stream

    def _launch(self, img_hw, shift_corners):
        lib, B, P = self.lib, self.B, self.P
        # cat((a, b), dim=1) (model.py:96): the two patches are the two channels of the static NCHW input pair, packed
        # into the 16-channel-pitch NHWC bf16 buffer the first conv reads (channels 2..15 stay zero)
        ops.nchw_to_nhwc_into(self.ab, self.x_in)
        for _, fn in self.steps:
            fn()
        k1 = self.w1.shape[1]
        check(lib.masic_fc_bf16(self.feat.data_ptr(), k1, self.w1.data_ptr(), self.b1.data_ptr(), B, k1, 1024, 1, None,
                                self.h1.data_ptr(), 1024, F16, self._s()), "masic_fc_bf16")
        check(lib.masic_fc_bf16(self.h1.data_ptr(), 1024, self.w2.data_ptr(), self.b2.data_ptr(), B, 1024, 8, 0,
                                self.delta.data_ptr(), None, 8, F16, self._s()), "masic_fc_bf16")
        if img_hw is not None:
            check(lib.masic_homography_from_delta(self.corners.data_ptr(), self.delta.data_ptr(), B, int(shift_corners),
                                                  img_hw[0], img_hw[1], PIC_SIZE, PIC_SIZE, self.h.data_ptr(), self._s()),
                  "masic_homography_from_delta")

    @property
    def ab(self) -> torch.Tensor:
        """(B, 2, P, P) fp32 static input: channel 0 = patch a, channel 1 = patch b."""
        if getattr(self, "_ab", None) is None:
            self._ab = torch.zeros(self.B, 2, self.P, self.P, device=self.dev)
        return self._ab

    def run(self, a: Optional[torch.Tensor] = None, b: Optional[torch.Tensor] = None,
            corners: Optional[torch.Tensor] = None, img_hw: Optional[Tuple[int, int]] = None,
            shift_corners: bool = True) -> Dict[str, torch.Tensor]:
        """Copies the inputs into the static buffers and replays the graph.  Returns {'delta', 'h'} (static buffers)."""
        with torch.cuda.device(self.dev):
            if a is not None:
                self.ab[:, 0:1].copy_(a.reshape(self.B, 1, self.P, self.P), non_blocking=True)
            if b is not None:
                self.ab[:, 1:2].copy_(b.reshape(self.B, 1, self.P, self.P), non_blocking=True)
            want_h = img_hw is not None and corners is not None
            if want_h:
                self.corners.copy_(corners.reshape(self.B, 4, 2), non_blocking=True)
            key = (tuple(img_hw), bool(shift_corners)) if want_h else None
            args = (key[0], key[1]) if want_h else (None, True)
            if not self.use_graph:
                self._launch(*args)
            else:
                if self.graph is None or self._graph_key != key:
                    self._launch(*args)                         # warm-up outside capture
                    torch.cuda.synchronize(self.dev)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._launch(*args)
                    self.graph, self._graph_key = g, key
                self.graph.replay()
        return {"delta": self.delta, "h": self.h}
