"""Pairs of any size (masic_b200/padding.py), the parts that need no GPU: the padded frame against CompressAI's
evaluation rule, the homography algebra of the padded frame, the bitstream header of odd sizes and its size limit, and
the argument checks of the two new C entry points."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from masic_b200 import _lib
from masic_b200.build import build
from masic_b200.padding import HEADER_MAX, padding_for

SIZES = [1, 2, 31, 63, 64, 65, 100, 127, 128, 129, 130, 200, 333, 375, 860, 1080, 1242, 2176]


def _compressai(h, w, p=64):
    """compressai/utils/eval_model/__main__.py, inference(): new size and F.pad's (left, right, top, bottom)."""
    new_h = (h + p - 1) // p * p
    new_w = (w + p - 1) // p * p
    padding_left = (new_w - w) // 2
    padding_right = new_w - w - padding_left
    padding_top = (new_h - h) // 2
    padding_bottom = new_h - h - padding_top
    return new_h, new_w, (padding_left, padding_right, padding_top, padding_bottom)


@pytest.mark.parametrize("h", SIZES)
def test_padded_frame_is_compressais(h):
    for w in SIZES:
        pad = padding_for(h, w)
        new_h, new_w, args = _compressai(h, w)
        assert (pad.hp, pad.wp) == (new_h, new_w)
        assert pad.pad_args() == args
        assert (pad.left, pad.top) == (args[0], args[2])
        assert pad.aligned == (h % 64 == 0 and w % 64 == 0)


def test_pad_and_crop_round_trip():
    g = torch.Generator().manual_seed(0)
    for h, w in ((1, 1), (63, 65), (375, 1242), (64, 128)):
        pad = padding_for(h, w)
        x = torch.rand(2, 3, h, w, generator=g)
        xp = F.pad(x, pad.pad_args(), mode="constant", value=0)
        assert xp.shape == (2, 3, pad.hp, pad.wp)
        assert torch.equal(pad.crop(xp), x)
        border = xp.clone()
        pad.crop(border).zero_()
        assert not border.any()                                  # everything outside the window is padding


def test_invalid_sizes():
    for h, w in ((0, 10), (10, 0), (-1, 5)):
        with pytest.raises(ValueError):
            padding_for(h, w)


def test_homography_of_the_padded_frame():
    """A pixel mapped through T H T^-1 in the padded frame lands at T(H p): the warp of the padded pair is the warp of
    the pair, moved by the padding offset (float64 numpy)."""
    rng = np.random.default_rng(5)
    for h, w in ((375, 1242), (200, 333), (100, 130), (1, 63)):
        pad = padding_for(h, w)
        T = np.array([[1, 0, pad.left], [0, 1, pad.top], [0, 0, 1]], dtype=np.float64)
        H = np.eye(3) + rng.normal(scale=[[0.05, 0.05, 5], [0.05, 0.05, 5], [1e-4, 1e-4, 0]], size=(3, 3))
        Hp = T @ H @ np.linalg.inv(T)
        for _ in range(20):
            p = np.array([rng.uniform(0, w), rng.uniform(0, h), 1.0])
            q = H @ p
            q /= q[2]
            r = Hp @ (T @ p)
            r /= r[2]
            np.testing.assert_allclose(r[:2], q[:2] + [pad.left, pad.top], rtol=0, atol=1e-9)


def _header(h, w, M=192):
    from masic_b200.bitstream import _header_bytes
    rng = np.random.default_rng(h * 7 + w)
    flags = [rng.integers(0, 2, M), rng.integers(0, 2, M)]
    return _header_bytes(h, w, [b"\x01\x02\x03", b""], [3, 1], flags), flags


@pytest.mark.parametrize("hw", [(375, 1242), (1, 1), (63, 65), (860, 1080), (HEADER_MAX - 63, 64)])
def test_header_keeps_the_original_size(hw):
    from masic_b200.bitstream import _header_padding, _parse_header
    data, flags = _header(*hw)
    H, W, views = _parse_header(data, 192)
    assert (H, W) == hw
    assert views[0][0] == b"\x01\x02\x03" and views[1][0] == b""
    assert all(np.array_equal(v[2], f) for v, f in zip(views, flags))
    pad = _header_padding(H, W)
    assert (pad.hp, pad.wp) == (padding_for(*hw).hp, padding_for(*hw).wp)


def test_size_limit():
    from masic_b200.bitstream import _header_padding
    from masic_b200.hsic import HSIC
    padding_for(HEADER_MAX - 63, HEADER_MAX - 63).check_header()      # pads to 65472: fits
    for h, w in ((HEADER_MAX - 62, 10), (10, HEADER_MAX)):
        with pytest.raises(ValueError):
            padding_for(h, w).check_header()
        with pytest.raises(_lib.MasicError):
            _header_padding(h, w)                                        # a header no encoder writes
    with pytest.raises(_lib.MasicError):
        _header_padding(0, 64)
    x = torch.zeros(1, 3, HEADER_MAX - 62, 1)
    with pytest.raises(ValueError):
        HSIC().eval().compress(x, x, torch.eye(3)[None], "unused")      # refused before anything runs


@pytest.fixture(scope="module")
def lib():
    build()
    return _lib.load()


def test_new_entry_points_reject_bad_arguments(lib):
    buf = (np.zeros(64, np.float32)).ctypes.data
    assert lib.masic_pad_image(None, 1, 1, 3, 4, 4, 64, 64, 0, 0, buf, None, None) == -1
    assert lib.masic_pad_image(buf, 1, 1, 3, 4, 4, 64, 64, 0, 0, None, None, None) == -1
    assert lib.masic_pad_image(buf, 1, 1, 3, 4, 4, 64, 64, 61, 0, buf, None, None) == -1   # window outside the frame
    assert lib.masic_pad_image(buf, 1, 1, 3, 4, 4, 64, 64, 0, -1, buf, None, None) == -1
    assert lib.masic_pad_image(buf, 1, 0, 3, 4, 4, 64, 64, 0, 0, buf, None, None) == -1
    assert lib.masic_homography_pad(None, 1, 0, 0, buf, None) == -1
    assert lib.masic_homography_pad(buf, 0, 0, 0, buf, None) == -1
