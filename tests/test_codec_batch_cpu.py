"""CPU-side checks of the batched coding entry points: NULL pointers, negative counts and misaligned channel counts
are rejected with MASIC_EINVAL before anything touches a device (the fake pointers below are never dereferenced)."""
import pytest

from masic_b200 import _lib
from masic_b200.build import build

EINVAL = -1
P = 0x1000            # a non-NULL pointer that must never be dereferenced


@pytest.fixture(scope="module")
def lib():
    build()
    return _lib.load()


def _cdfs(lib, **kw):
    a = dict(sigma=P, mu=P, w=P, logits=1, m=192, k=5, n_pos=4, pair_stride=4, pair=P, ch=P, mm=P, n_streams=2,
             max_minmax=3, bound=0.11, y=P, rows=P, pitch=8, iv=P)
    a.update(kw)
    return lib.masic_gmm_symbol_cdfs_pairs(*a.values(), None)


def _gather(lib, **kw):
    a = dict(ypad=P, h16=4, w16=8, m=192, gmm=P, cin=960, c_lo=384, c_hi0=768, mw=P, pos=P, n=3, n_pairs=2, n_max=4,
             crop=P, rs=P, px=P)
    a.update(kw)
    return lib.masic_wave_gather_pairs(*a.values(), None)


def _decode(lib, **kw):
    a = dict(rows=P, n=3, n_streams=2, pitch=8, state=P, data=P, offs=P, pair=P, ch=P, mm=P, max_minmax=3, pos=P,
             h16=4, w16=8, m=192, y=P, ypad=P, f16=1, err=P)
    a.update(kw)
    return lib.masic_range_decode_wave_pairs(*a.values(), None)


def _encode(lib, **kw):
    a = dict(iv=P, base=P, stride=P, n_pos=10, n_streams=2, slots=P, slot_cap=46, lens=P, err=P)
    a.update(kw)
    return lib.masic_range_encode_streams(*a.values(), None)


def _pack(lib, **kw):
    a = dict(slots=P, slot_cap=46, lens=P, n_streams=2, offs=P, packed=P)
    a.update(kw)
    return lib.masic_pack_streams(*a.values(), None)


@pytest.mark.parametrize("bad", [dict(sigma=None), dict(mu=None), dict(w=None), dict(pair=None), dict(ch=None),
                                 dict(mm=None), dict(rows=None, iv=None), dict(y=None), dict(m=0), dict(n_pos=-1),
                                 dict(pair_stride=-1), dict(n_streams=-1), dict(max_minmax=0),
                                 dict(max_minmax=40000, pitch=80002), dict(pitch=7)])
def test_symbol_cdfs_pairs_rejects_bad_arguments(lib, bad):
    assert _cdfs(lib, **bad) == EINVAL


@pytest.mark.parametrize("bad", [dict(ypad=None), dict(gmm=None), dict(pos=None), dict(crop=None), dict(px=None),
                                 dict(mw=None), dict(h16=0), dict(w16=-1), dict(m=0), dict(cin=0), dict(n=-1),
                                 dict(n_pairs=0), dict(n_pairs=-2), dict(n_max=2), dict(m=20), dict(cin=964),
                                 dict(c_lo=4), dict(c_hi0=770)])
def test_wave_gather_pairs_rejects_bad_arguments(lib, bad):
    assert _gather(lib, **bad) == EINVAL


@pytest.mark.parametrize("bad", [dict(rows=None), dict(state=None), dict(data=None), dict(offs=None), dict(pair=None),
                                 dict(ch=None), dict(mm=None), dict(pos=None), dict(y=None), dict(ypad=None),
                                 dict(err=None), dict(n=-1), dict(n_streams=-1), dict(max_minmax=0), dict(pitch=7),
                                 dict(h16=0), dict(w16=0), dict(m=-8)])
def test_range_decode_wave_pairs_rejects_bad_arguments(lib, bad):
    assert _decode(lib, **bad) == EINVAL


@pytest.mark.parametrize("bad", [dict(iv=None), dict(base=None), dict(stride=None), dict(slots=None), dict(lens=None),
                                 dict(err=None), dict(n_pos=-1), dict(n_streams=-1), dict(slot_cap=45)])
def test_range_encode_streams_rejects_bad_arguments(lib, bad):
    assert _encode(lib, **bad) == EINVAL


@pytest.mark.parametrize("bad", [dict(slots=None), dict(lens=None), dict(offs=None), dict(packed=None),
                                 dict(slot_cap=0), dict(n_streams=-1)])
def test_pack_streams_rejects_bad_arguments(lib, bad):
    assert _pack(lib, **bad) == EINVAL


def test_empty_calls_launch_nothing(lib):
    """Zero streams or zero positions are empty calls: they return before any launch, so they succeed here too."""
    assert _cdfs(lib, n_streams=0) == 0
    assert _cdfs(lib, n_pos=0) == 0
    assert _gather(lib, n=0) == 0
    assert _decode(lib, n_streams=0) == 0
    assert _decode(lib, n=0) == 0
    assert _encode(lib, n_streams=0) == 0
