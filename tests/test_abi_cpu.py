"""CPU-side checks of the C-ABI boundary: the library loads without a GPU, exports every
symbol include/masic_b200.h declares, rejects bad arguments with its error codes, and its
host-side integer code (pmf -> cdf) reproduces the reference's known answers."""
import ctypes as C
import json
import re
import subprocess

import numpy as np
import pytest

from masic_b200 import _lib, ops
from masic_b200.build import build


@pytest.fixture(scope="module")
def lib():
    build()
    return _lib.load()


def _header_symbols(root):
    hdr = (root / "include" / "masic_b200.h").read_text()
    return sorted(set(re.findall(r"\b(masic_[a-z0-9_]+)\s*\(", hdr)))


def test_library_matches_the_header_and_abi_version(lib):
    ROOT = _lib.LIB_PATH.parents[1]
    names = _header_symbols(ROOT)
    assert len(names) >= 25
    out = subprocess.run(["nm", "-D", "--defined-only", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True)
    exported = {ln.split()[-1] for ln in out.stdout.splitlines() if ln.strip()}
    missing = [n for n in names if n not in exported]
    assert not missing, missing
    assert sorted(_lib.declared_symbols()) == names          # the ctypes binding covers the whole header
    assert lib.masic_abi_version() == 11
    assert b"sm_100a" in lib.masic_build_info()


def test_only_sm100a_code_in_the_binary():
    out = subprocess.run(["cuobjdump", "-lelf", str(_lib.LIB_PATH)], capture_output=True, text=True)
    archs = set(re.findall(r"sm_(\d+a?)", out.stdout))
    assert archs == {"100a"}, archs


def test_bad_arguments_are_rejected_without_a_gpu(lib):
    d = _lib.ConvDesc()
    h = C.c_void_p()
    assert lib.masic_conv_plan_create(None, C.byref(h)) == -1
    d.c_in = 10                                    # not a multiple of 16
    assert lib.masic_conv_plan_create(C.byref(d), C.byref(h)) == -1
    assert lib.masic_gmm_likelihood_fwd(None, None, None, None, 0, 0, 1, 1, 5, 1, 0.11, None, None, None, 0,
                                        None, 0, 0, None, 0, 0, 0, None) == -1
    assert lib.masic_conv_plan_launch(None, None) == -1
    assert lib.masic_pmf_to_quantized_cdf(None, 3, 16, None) == -1


def test_pmf_to_cdf_kats(lib, golden_dir):
    kat = json.loads((golden_dir / "pmf_cdf_kat.json").read_text())
    for c in kat["cases"]:
        if "error" in c:
            with pytest.raises(ValueError):
                ops.pmf_to_quantized_cdf(c["pmf"], kat["precision"])
        else:
            assert ops.pmf_to_quantized_cdf(c["pmf"], kat["precision"]) == c["cdf"]
    for bad in ([-0.1, 0.5], [float("nan"), 1.0], [0.0, 0.0]):
        with pytest.raises(ValueError):
            ops.pmf_to_quantized_cdf(bad)


def test_pmf_to_cdf_random_against_oracle(lib):
    from oracle import entropy as E
    rng = np.random.default_rng(3)
    for _ in range(200):
        p = rng.random(int(rng.integers(1, 100))).astype(np.float32) ** int(rng.integers(1, 10))
        if p.sum() * 65536 < 1:
            continue
        assert ops.pmf_to_quantized_cdf(p) == [int(v) for v in E.pmf_to_quantized_cdf_c(p)]


def test_cuda_ops_refuse_cpu_tensors():
    import torch
    with pytest.raises(_lib.MasicError):
        ops.quantize(torch.zeros(4))
    with pytest.raises(_lib.MasicError):
        ops.gmm_likelihood(torch.zeros(1, 2, 2, 2), torch.zeros(1, 10, 2, 2), torch.zeros(1, 10, 2, 2),
                           torch.zeros(1, 10, 2, 2))


def test_torch_library_custom_ops_are_registered_with_fake_impls():
    """SURVEY §8(b) / north-star: "thin C-ABI torch custom-op extension" — every op is a torch.ops.masic_b200.* custom
    op with a schema and a fake (meta) implementation; CPU tensors are refused (no fallback)."""
    import torch
    from masic_b200 import torch_ops
    for name in torch_ops.OPS:
        op = getattr(torch.ops.masic_b200, name)
        assert op.default._schema.name == f"masic_b200::{name}"
    m = lambda *s: torch.empty(*s, device="meta")   # noqa: E731
    assert torch.ops.masic_b200.conv2d(m(2, 128, 64, 96), m(128, 128, 5, 5), m(128), 2, False, 0).shape == (2, 128, 32, 48)
    assert torch.ops.masic_b200.conv2d(m(2, 128, 64, 96), m(128, 3, 5, 5), None, 2, True, 0).shape == (2, 3, 128, 192)
    assert torch.ops.masic_b200.gdn(m(1, 128, 8, 8), m(128), m(128, 128), False, 1e-6).shape == (1, 128, 8, 8)
    assert torch.ops.masic_b200.warp_perspective(m(1, 3, 64, 64), m(1, 3, 3), 32, 48).shape == (1, 3, 32, 48)
    y_hat, lik = torch.ops.masic_b200.gmm_likelihood(m(1, 192, 4, 4), m(1, 960, 4, 4), m(1, 960, 4, 4), m(1, 960, 4, 4), 0.11)
    assert y_hat.shape == lik.shape == (1, 192, 4, 4)
    assert torch.ops.masic_b200.gc_build_indexes(m(1, 8, 4, 4), m(64), 0.11).dtype == torch.int32
    assert torch.ops.masic_b200.quantize(m(1, 8, 4, 4), None, True).dtype == torch.int32
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.masic_b200.gdn(torch.zeros(1, 3, 4, 4), torch.ones(3), torch.eye(3), False, 1e-6)     # CPU: no kernel
