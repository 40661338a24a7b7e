"""HSIC.compress_batch / decompress_batch: the device range encoder byte for byte against the host encoder, the batch
payloads against a per-pair reference assembled without the batch path, the batch decoder against per-pair decoding
and forward(), file interop both ways, and the error paths."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

M = 192


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def net(dev):
    from masic_b200.hsic import HSIC
    torch.manual_seed(0)
    n = HSIC().eval()
    with torch.no_grad():
        n.encoder1.g_a_conv4.weight.mul_(8.0)          # non-degenerate latents (SURVEY §8d): at init every y symbol is 0
        n.encoder2.g_a_conv4.weight.mul_(8.0)
    n = n.to(dev)
    n.update(force=True)
    return n


def _pairs(B, h, w, seed, dev, kinds=(0, 1, 2, 3)):
    """B pairs of different content, pair b of kind kinds[b % len(kinds)]: 0 noise, 1 low-contrast noise, 2 smooth
    ramps, 3 flat images, 4 noise of three times the image range (larger latents)."""
    g = torch.Generator().manual_seed(seed)
    xs = []
    for b in range(B):
        kind = kinds[b % len(kinds)]
        if kind == 0:
            x = torch.rand(2, 3, h, w, generator=g)
        elif kind == 1:
            x = 0.5 + 0.08 * torch.rand(2, 3, h, w, generator=g)
        elif kind == 2:
            ramp = torch.linspace(0, 1, w).view(1, 1, 1, w) * torch.linspace(0.2, 0.9, h).view(1, 1, h, 1)
            x = ramp.expand(2, 3, h, w) * torch.rand(2, 3, 1, 1, generator=g)
        elif kind == 3:
            x = torch.full((2, 3, h, w), 0.3) + 0.4 * torch.rand(2, 3, 1, 1, generator=g)
        else:
            x = 3.0 * torch.rand(2, 3, h, w, generator=g)
        xs.append(x)
    x = torch.stack(xs)                                     # (B, 2, 3, h, w)
    from oracle.hsic import synthetic_homography
    Hm = synthetic_homography(B, seed=seed)
    return x[:, 0].contiguous().to(dev), x[:, 1].contiguous().to(dev), Hm.to(dev)


def _reference_item(net, x1, x2, Hm):
    """Format-2 header and payload of ONE pair as the batch-1 path built them before the batch coder existed: the
    batch-1 engine's intervals (one `masic_gmm_symbol_cdfs` call per view), wave order on the host, the host encoder
    `masic_range_encode_channels`."""
    from masic_b200 import _lib, bitstream as bs
    lib = _lib.load()
    _, _, H, W = x1.shape
    eng = net.engine_for(1, H, W, x1.device)
    out = eng.run(x1, x2, Hm)
    n_pos = (H // 16) * (W // 16)
    perm = bs.wave_permutation(H // 16, W // 16)
    header = [np.array([H, W], dtype=np.uint16).tobytes()]
    payload = [bytes([2])]
    stats = []
    for tag, eb, yk in (("L", net.entropy_bottleneck1, "y1_hat"), ("R", net.entropy_bottleneck2, "y2_hat")):
        zs = eb.compress(eng.buf[f"{tag}.z"].permute(0, 3, 1, 2).contiguous())[0]
        flag, minmax = bs._nonzero_channels(out[yk])
        header += [np.array([len(zs), minmax], dtype=np.uint16).tobytes(), bs._pack_flags(flag), zs]
        n_ch = int(flag.sum())
        payload.append(np.array([n_ch], dtype=np.uint32).tobytes())
        stats.append((minmax, flag.copy()))
        if n_ch:
            ch = torch.from_numpy(np.flatnonzero(flag).astype(np.int32)).to(x1.device)
            a = bs._symbol_intervals(eng, tag, out[yk], ch, minmax)
            a = np.ascontiguousarray(a.reshape(n_pos, n_ch, 3)[perm])
            buf = np.empty(a.size + 16 * n_ch + 64, dtype=np.uint8)
            lens = np.zeros(n_ch, dtype=np.int64)
            _lib.check(lib.masic_range_encode_channels(a.ctypes.data, n_pos, n_ch, buf.ctypes.data, buf.size,
                                                       lens.ctypes.data), "masic_range_encode_channels")
            payload += [lens.astype(np.uint32).tobytes(), buf[:int(lens.sum())].tobytes()]
    return b"".join(header), b"".join(payload), stats


# ---------------------------------------------------------------------------------------------- the device encoder
def _gpu_encode(lib, iv_np, base, stride, n_pos, dev):
    from masic_b200 import _lib
    S = len(base)
    iv = torch.from_numpy(np.ascontiguousarray(iv_np, dtype=np.int32).reshape(-1)).to(dev)
    if iv.numel() == 0:
        iv = torch.zeros(3, dtype=torch.int32, device=dev)
    cap = 3 * n_pos + 16
    slots = torch.zeros(max(S, 1) * cap, dtype=torch.uint8, device=dev)
    packed = torch.zeros_like(slots)
    lens = torch.zeros(max(S, 1), dtype=torch.int64, device=dev)
    offs = torch.zeros(S + 1, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    b = torch.tensor(base, dtype=torch.int64, device=dev)
    s = torch.tensor(stride, dtype=torch.int64, device=dev)
    _lib.check(lib.masic_range_encode_streams(iv.data_ptr(), b.data_ptr(), s.data_ptr(), n_pos, S, slots.data_ptr(),
                                              cap, lens.data_ptr(), err.data_ptr(), None), "masic_range_encode_streams")
    _lib.check(lib.masic_pack_streams(slots.data_ptr(), cap, lens.data_ptr(), S, offs.data_ptr(), packed.data_ptr(),
                                      None), "masic_pack_streams")
    o = offs.cpu().numpy()
    return int(err.item()), packed[:int(o[-1])].cpu().numpy().tobytes(), np.diff(o)


def _host_encode(lib, iv_np, n_pos, n_ch):
    a = np.ascontiguousarray(iv_np, dtype=np.int32)
    buf = np.empty(3 * n_pos * n_ch + 16 * n_ch + 64, dtype=np.uint8)
    lens = np.zeros(n_ch, dtype=np.int64)
    rc = lib.masic_range_encode_channels(a.ctypes.data if a.size else None, n_pos, n_ch, buf.ctypes.data, buf.size,
                                         lens.ctypes.data)
    return rc, buf[:int(lens.sum())].tobytes(), lens


def _random_intervals(rng, n_pos, n_ch, mode):
    total = rng.integers(1, (1 << 22) + 1, size=(n_pos, n_ch))
    total[rng.random((n_pos, n_ch)) < 0.1] = 1 << 22
    if mode == "top":        # the top end of every range: low creeps upwards
        freq = np.maximum(1, total // rng.integers(1, 4, size=total.shape))
        cum = total - freq
    else:
        freq = rng.integers(1, total + 1)
        freq[rng.random(total.shape) < 0.2] = 1
        cum = (rng.random(total.shape) * (total - freq + 1)).astype(np.int64)
    return np.stack([cum, freq, total], -1).astype(np.int32)


@pytest.mark.parametrize("n_pos,n_ch,mode", [(0, 3, "mix"), (1, 1, "mix"), (1, 40, "top"), (2000, 1, "mix"),
                                             (2000, 1, "top"), (1500, 37, "mix"), (1500, 37, "top")])
def test_device_encoder_is_byte_identical_to_the_host_encoder(dev, n_pos, n_ch, mode):
    from masic_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(n_pos * 7 + n_ch + (mode == "top"))
    iv = _random_intervals(rng, n_pos, n_ch, mode)
    if mode == "top" and n_pos > 1:
        # the top symbol of the largest total, freq 1: low stays just below a byte boundary, so byte after byte is
        # held back as a pending 0xFF (a long carry run); then the same symbol at every other position
        iv[: n_pos // 2] = [(1 << 22) - 1, 1, 1 << 22]
        iv[n_pos // 2 + 1::2] = [(1 << 22) - 1, 1, 1 << 22]
    rc, host, host_lens = _host_encode(lib, iv, n_pos, n_ch)
    assert rc == 0
    err, gpu, gpu_lens = _gpu_encode(lib, iv, list(range(n_ch)), [n_ch] * n_ch, n_pos, dev)
    assert err == 0
    assert np.array_equal(gpu_lens, host_lens)
    assert gpu == host
    if mode == "top" and n_pos > 1:
        assert b"\xff" * 8 in host or b"\x00" * 8 in host    # a run of held-back bytes was released


def test_device_encoder_reads_blocks_by_base_and_stride(dev):
    """Two (n_pos, n_ch, 3) blocks in one buffer, encoded by one launch, equal each block encoded on the host."""
    from masic_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(11)
    n_pos = 300
    a, b = _random_intervals(rng, n_pos, 5, "mix"), _random_intervals(rng, n_pos, 3, "top")
    buf = np.concatenate([a.reshape(-1), b.reshape(-1)])
    err, gpu, lens = _gpu_encode(lib, buf, [0, 1, 2, 3, 4, n_pos * 5, n_pos * 5 + 1, n_pos * 5 + 2], [5] * 5 + [3] * 3,
                                 n_pos, dev)
    _, ha, la = _host_encode(lib, a, n_pos, 5)
    _, hb, lb = _host_encode(lib, b, n_pos, 3)
    assert err == 0 and gpu == ha + hb and np.array_equal(lens, np.concatenate([la, lb]))


@pytest.mark.parametrize("field,value", [(0, -1), (1, 0), (1, -3), (0, 90), (2, (1 << 22) + 1)])
def test_device_encoder_flags_what_the_host_encoder_rejects(dev, field, value):
    from masic_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    iv = _random_intervals(rng, 50, 4, "mix")
    iv[17, 2] = [60, 20, 100]
    iv[17, 2, field] = value
    rc, _, _ = _host_encode(lib, iv, 50, 4)
    assert rc == -1
    err, _, _ = _gpu_encode(lib, iv, [0, 1, 2, 3], [4] * 4, 50, dev)
    assert err == 1


# ---------------------------------------------------------------------------------------------- batch encoder
def _mixed(stats):
    """Whether the batch mixes pairs with different minmax and different non-zero-channel bitmaps in one view."""
    return any(len({s[v][0] for s in stats}) > 1 and len({s[v][1].tobytes() for s in stats}) > 1 for v in range(2))


@pytest.mark.parametrize("B,h,w", [(1, 192, 256), (3, 192, 256), (4, 192, 256), (2, 1216, 2176)])
def test_compress_batch_bytes_equal_the_per_pair_reference(net, dev, B, h, w):
    # at 1216x2176 every in-range content gives the same minmax (2 and 1): the first pairing of contents that differs
    # in minmax and bitmap is used
    for kinds in ((0, 1, 2, 3), (0, 4), (3, 4), (1, 4)):
        x1, x2, Hm = _pairs(B, h, w, seed=B, dev=dev, kinds=kinds)
        with torch.no_grad():
            ref = [_reference_item(net, x1[b:b + 1], x2[b:b + 1], Hm[b:b + 1]) for b in range(B)]
        if B == 1 or _mixed([r[2] for r in ref]):
            break
    else:
        raise AssertionError(f"no batch mixes minmax and bitmaps: {[(r[2][0][0], r[2][1][0]) for r in ref]}")
    with torch.no_grad():
        items = net.compress_batch(x1, x2, Hm)
    assert len(items) == B
    for b, (it, (hdr, pay, _)) in enumerate(zip(items, ref)):
        assert it["header"] == hdr, f"pair {b}: header"
        assert it["payload"] == pay, f"pair {b}: payload"
        assert it["bpp_real"] == (len(hdr) + len(pay)) * 8 / (2 * h * w)
        assert it["n_symbols"] > 0 and it["y_bits_ideal"] > 0
        assert len(pay) * 8 >= it["y_bits_ideal"]


def test_compress_batch_raises_on_an_invalid_interval(net, dev, monkeypatch):
    from masic_b200 import bitstream as bs
    from masic_b200._lib import MasicError
    orig = bs._stream_intervals

    def corrupt(eng, tag, y, table, mm, out):
        orig(eng, tag, y, table, mm, out)
        out[3, 0, 1] = 0                                   # an empty interval
    monkeypatch.setattr(bs, "_stream_intervals", corrupt)
    x1, x2, Hm = _pairs(2, 192, 256, seed=9, dev=dev)
    with torch.no_grad(), pytest.raises(MasicError, match="invalid coding interval"):
        net.compress_batch(x1, x2, Hm)


# ---------------------------------------------------------------------------------------------- batch decoder
def _per_pair(net, x1, x2, Hm, tmp_path):
    """forward() and compress / decompress of every pair through the file API."""
    res = []
    with torch.no_grad():
        for b in range(x1.shape[0]):
            fwd = net(x1[b:b + 1], x2[b:b + 1], Hm[b:b + 1])
            enc = net.compress(x1[b:b + 1], x2[b:b + 1], Hm[b:b + 1], f"p{b}", str(tmp_path))
            dec = net.decompress(None, None, Hm[b:b + 1], f"p{b}", str(tmp_path), device=x1.device)
            res.append((fwd, enc, dec))
    return res


def _read(tmp_path, name):
    return (tmp_path / f"{name}.npz").read_bytes(), (tmp_path / f"{name}.bin").read_bytes()


KEYS = ("x1_hat", "x2_hat", "y1_hat", "y2_hat", "z1_hat", "z2_hat")


def _header_stats(header):
    """[(minmax, bitmap)] of the two views, as `_reference_item` reports them."""
    from masic_b200 import bitstream as bs
    return [(mm, flag) for _, mm, flag in bs._parse_header(header, M)[2]]


def test_decompress_batch_equals_per_pair_decompress_and_forward(net, dev, tmp_path):
    B = 4
    x1, x2, Hm = _pairs(B, 192, 256, seed=21, dev=dev, kinds=(0, 4, 2, 3))
    per = _per_pair(net, x1, x2, Hm, tmp_path)
    for fwd, enc, dec in per:
        for k in ("x1_hat", "x2_hat", "y1_hat", "z1_hat"):
            assert torch.equal(dec[k], fwd[k]), k
        for k in ("y2_hat", "z2_hat"):
            assert torch.equal(dec[k], enc[k]), k
    with torch.no_grad():
        items = net.compress_batch(x1, x2, Hm)
    # the batch decoder sees streams of different minmax (row lengths inside one row pitch) and bitmaps
    assert _mixed([_header_stats(it["header"]) for it in items])
    for order in ([0, 1, 2, 3], [2, 0, 3, 1]):
        with torch.no_grad():
            out = net.decompress_batch([(items[i]["header"], items[i]["payload"]) for i in order], Hm[order])
        for j, i in enumerate(order):
            for k in KEYS:
                assert torch.equal(out[k][j:j + 1], per[i][2][k]), (order, i, k)


def test_files_and_batch_bytes_interoperate(net, dev, tmp_path):
    B = 3
    x1, x2, Hm = _pairs(B, 192, 256, seed=33, dev=dev)
    per = _per_pair(net, x1, x2, Hm, tmp_path)
    with torch.no_grad():
        out = net.decompress_batch([_read(tmp_path, f"p{b}") for b in range(B)], Hm)     # files -> batch decoder
        items = net.compress_batch(x1, x2, Hm)
    for b in range(B):
        for k in KEYS:
            assert torch.equal(out[k][b:b + 1], per[b][2][k]), (b, k)
        (tmp_path / f"q{b}.npz").write_bytes(items[b]["header"])                             # batch bytes -> files
        (tmp_path / f"q{b}.bin").write_bytes(items[b]["payload"])
        with torch.no_grad():
            dec = net.decompress(None, None, Hm[b:b + 1], f"q{b}", str(tmp_path), device=dev)
        for k in KEYS:
            assert torch.equal(dec[k], per[b][2][k]), (b, k)


def _drop_view(header, payload, v):
    """The same pair with view v coded as having no non-zero channel (bitmap cleared, empty stream table)."""
    from masic_b200 import bitstream as bs
    _, _, views = bs._parse_header(header, M)
    streams = bs._parse_payload(payload, views)
    hdr = bytearray(header)
    p = 4 + (4 + M // 8 + len(views[0][0])) * v
    hdr[p + 4:p + 4 + M // 8] = bytes(M // 8)
    parts = [bytes([2])]
    for u, (lens, data) in enumerate(streams):
        if u == v:
            parts.append(np.array([0], dtype=np.uint32).tobytes())
        else:
            parts += [np.array([lens.size], dtype=np.uint32).tobytes()] + \
                     ([lens.astype(np.uint32).tobytes(), data] if lens.size else [])
    return bytes(hdr), b"".join(parts)


def test_views_without_streams_next_to_views_with_streams(net, dev, tmp_path):
    """A view with no non-zero channel decodes to zeros beside pairs that have streams, and a batch with no stream at
    all (S = 0 for both views) decodes too; every pair equals its own decode through the file API."""
    B = 3
    x1, x2, Hm = _pairs(B, 192, 256, seed=44, dev=dev)
    with torch.no_grad():
        items = net.compress_batch(x1, x2, Hm)
    base = [(it["header"], it["payload"]) for it in items]
    # only right views are dropped next to full pairs: the right view's CDFs depend on the left view's decode (through
    # round(y1warp) * w2), so a pair whose left view is cleared but whose right streams are kept is not a valid pair
    mixed = [base[0], _drop_view(*base[1], 1), _drop_view(*base[2], 1)]
    empty = [_drop_view(*_drop_view(*it, 0), 1) for it in base]
    for batch in (mixed, empty):
        with torch.no_grad():
            out = net.decompress_batch(batch, Hm)
        for b, (hdr, pay) in enumerate(batch):
            (tmp_path / f"d{b}.npz").write_bytes(hdr)
            (tmp_path / f"d{b}.bin").write_bytes(pay)
            with torch.no_grad():
                dec = net.decompress(None, None, Hm[b:b + 1], f"d{b}", str(tmp_path), device=dev)
            for k in KEYS:
                assert torch.equal(out[k][b:b + 1], dec[k]), (b, k)
    assert not out["y1_hat"].any() and not out["y2_hat"].any()
    with torch.no_grad():
        out = net.decompress_batch(mixed, Hm)
    assert not out["y2_hat"][1].any() and not out["y2_hat"][2].any()
    assert out["y1_hat"][1].any() and out["y1_hat"][2].any() and out["y2_hat"][0].any()


# ---------------------------------------------------------------------------------------------- errors
def test_error_paths(net, dev, monkeypatch):
    from masic_b200._lib import MasicError
    x1, x2, Hm = _pairs(2, 192, 256, seed=55, dev=dev)
    with torch.no_grad():
        items = net.compress_batch(x1, x2, Hm)
    good = [(it["header"], it["payload"]) for it in items]
    hdr, pay = good[0]
    with torch.no_grad():
        with pytest.raises(MasicError):                                     # truncated
            net.decompress_batch([good[1], (hdr, pay[:-7])], Hm)
        flipped = bytearray(pay)
        n_ch = int(np.frombuffer(pay[1:5], dtype=np.uint32)[0])
        p = 5 + 4 * n_ch
        for s in np.frombuffer(pay[5:5 + 4 * n_ch], dtype=np.uint32)[:8]:  # a flipped bit in each of 8 streams
            flipped[p + int(s) // 2] ^= 0x10
            p += int(s)
        with pytest.raises(MasicError, match="corrupt"):
            net.decompress_batch([good[1], (hdr, bytes(flipped))], Hm)
        for fmt in (0, 1):                                                  # single-pair formats
            with pytest.raises(MasicError, match="format 2"):
                net.decompress_batch([good[1], (hdr, bytes([fmt]) + pay[1:])], Hm)
        small = net.compress_batch(x1[:1, :, :128, :192].contiguous(), x2[:1, :, :128, :192].contiguous(), Hm[:1])
        with pytest.raises(ValueError):                                     # mixed sizes
            net.decompress_batch([good[0], (small[0]["header"], small[0]["payload"])], Hm)
        with pytest.raises(ValueError):                                     # h_matrix batch
            net.decompress_batch(good, Hm[:1])
        with pytest.raises(ValueError):
            net.compress_batch(x1, x2, Hm[:1])
        with pytest.raises(MasicError):                                     # CPU tensors
            net.compress_batch(x1.cpu(), x2.cpu(), Hm.cpu())
        with pytest.raises(MasicError):
            net.decompress_batch(good, Hm.cpu())
        monkeypatch.setattr(net.entropy_bottleneck2, "compress", lambda z: [b"\0" * 70000] * z.shape[0])
        with pytest.raises(MasicError, match="uint16 length field"):
            net.compress_batch(x1, x2, Hm)
        monkeypatch.undo()
    net.train()
    try:
        with pytest.raises(MasicError):
            net.compress_batch(x1, x2, Hm)
        with pytest.raises(MasicError):
            net.decompress_batch(good, Hm)
    finally:
        net.eval()
