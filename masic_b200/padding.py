"""Stereo pairs of any size.  The codec's networks need H and W to be multiples of 64 (y = x/16, z = y/4), so a pair of
size (h, w) is coded in a zero-padded frame and its reconstructions are cropped back, as CompressAI 1.2 evaluates
(compressai/utils/eval_model/__main__.py, inference()):

    p = 64;  Hp = ceil(h / p) * p,  Wp = ceil(w / p) * p
    top = (Hp - h) // 2,  left = (Wp - w) // 2          the rest of the padding goes to the bottom / right
    x_padded = F.pad(x, (left, Wp - w - left, top, Hp - h - top), mode="constant", value=0)

The warps inside the codec map pixel coordinates, so the homography of the padded frame is T H T^-1 with T the
translation by (left, top).  bpp divides by the pixel count of the original pair.

This module is the one place that knows the rule: forward, PairStream and the bitstream coder ask `padding_for(h, w)`
and use its offsets, pad, homography and crop.  A pair whose size is already a multiple of 64 has `aligned` set and
takes the unpadded path.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import ops

P = 64
HEADER_MAX = 65535          # the bitstream header stores H, W as uint16 (MASIC.py:922)


@dataclass(frozen=True)
class Padding:
    h: int
    w: int
    hp: int
    wp: int
    top: int
    left: int

    @property
    def aligned(self) -> bool:
        return self.hp == self.h and self.wp == self.w

    def pad_args(self):
        """The padding as F.pad's (left, right, top, bottom)."""
        return self.left, self.wp - self.w - self.left, self.top, self.hp - self.h - self.top

    def crop(self, t: torch.Tensor) -> torch.Tensor:
        """The (..., h, w) window of the original pair in a (..., hp, wp) tensor (a view)."""
        return t.narrow(-2, self.top, self.h).narrow(-1, self.left, self.w)

    def crop_into(self, padded: torch.Tensor, out: torch.Tensor) -> None:
        """Strided copy of the window into `out`, on the current stream."""
        out.copy_(self.crop(padded), non_blocking=True)

    def image_into(self, src: torch.Tensor, dst: torch.Tensor, unpadded=None) -> None:
        """src (n,c,h,w) uint8 (ToTensor's x / 255) or fp32 -> dst (n,c,hp,wp) fp32, border zeroed, on the current
        stream; `unpadded` (n,c,h,w) fp32, if given, receives the converted src."""
        ops.pad_image_into(src, dst, self.top, self.left, unpadded)

    def homography_into(self, h: torch.Tensor, out: torch.Tensor) -> None:
        """out (n,3,3) fp32 <- T h T^-1 (fp64 on the device, rounded once), on the current stream."""
        ops.homography_pad_into(h, out, self.top, self.left)

    def check_header(self) -> None:
        """Bitstreams store the original size and decode on the padded one: both must fit the header's uint16."""
        if self.hp > HEADER_MAX or self.wp > HEADER_MAX:
            raise ValueError(f"a {self.h}x{self.w} pair pads to {self.hp}x{self.wp}, which exceeds the bitstream "
                             f"header's uint16 size fields (at most {HEADER_MAX})")


def padding_for(h: int, w: int) -> Padding:
    """The padded frame of an (h, w) pair."""
    h, w = int(h), int(w)
    if h < 1 or w < 1:
        raise ValueError(f"a pair needs h, w >= 1, got {h}x{w}")
    hp, wp = -(-h // P) * P, -(-w // P) * P
    return Padding(h, w, hp, wp, (hp - h) // 2, (wp - w) // 2)


def run_engine(eng, pad: Padding, x1: torch.Tensor, x2: torch.Tensor, h_matrix: torch.Tensor):
    """One forward pass of the padded-size engine `eng` on the (B,3,h,w) pair: the inputs and the homography are padded
    into the engine's input buffers on the device.  Returns the engine's (padded) output buffers."""
    if pad.aligned:
        return eng.run(x1, x2, h_matrix)
    with torch.cuda.device(eng.dev):
        for src, dst in ((x1, eng.x1), (x2, eng.x2)):
            pad.image_into(ops._f32c(src.to(eng.dev)), dst)
        pad.homography_into(ops._f32c(h_matrix.reshape(eng.B, 3, 3).to(eng.dev)), eng.Hm)
        return eng.run()
