"""CQETrainer's host side without a GPU: the new entry points are exported and bound, and bad arguments raise before
anything reaches a device."""
import pytest
import torch

NEW_SYMBOLS = ("masic_conv_plan_set_act_out", "masic_act_bwd_bias_out", "masic_cqe_feature_fuse_bwd",
               "masic_cqe_blend_images_bwd")


def test_training_entry_points_exported_and_bound():
    from masic_b200 import _lib
    lib = _lib.load()
    declared = _lib.declared_symbols()
    for name in NEW_SYMBOLS:
        assert name in declared
        assert getattr(lib, name).argtypes
    assert lib.masic_abi_version() == 11


def test_new_entry_points_reject_bad_arguments():
    from masic_b200 import _lib
    lib = _lib.load()
    assert lib.masic_conv_plan_set_act_out(None, None, 64, 0) == -1
    assert lib.masic_act_bwd_bias_out(None, 64, 0, None, 64, 0, 2, 16, 64, None, 64, 0, None, None) == -1
    assert lib.masic_cqe_feature_fuse_bwd(None, 64, None, 32, None, 32, 32, None, None, 1, 8, 8, None, 32, None, 32,
                                          None, None) == -1
    assert lib.masic_cqe_blend_images_bwd(None, 16, None, None, 1, 8, 8, None, None) == -1


@pytest.mark.parametrize("h,w", [(60, 64), (64, 96), (0, 64)])
def test_trainer_rejects_sizes_the_codec_does_not_emit(h, w):
    from masic_b200.cqe import Independent_EN
    with pytest.raises(ValueError):
        Independent_EN().trainer(1, h, w, "cpu")


def test_trainer_has_no_cpu_fallback():
    from masic_b200._lib import MasicError
    from masic_b200.cqe import Independent_EN
    with pytest.raises(MasicError):
        Independent_EN().trainer(1, 64, 64, "cpu")


def test_parameter_count_and_order():
    """86 tensors, 1.56 M floats: the flat gradient buffer's size and named_parameters() order."""
    from masic_b200.cqe import Independent_EN
    names = [n for n, _ in Independent_EN().named_parameters()]
    assert len(names) == 86
    assert names[:2] == ["EBl1.RB1.conv1.weight", "EBl1.RB1.conv1.bias"]
    assert names[76:78] == ["conv2.weight", "conv2.bias"] and names[78].startswith("mask2weights_unit")
    n = sum(p.numel() for p in Independent_EN().parameters())
    assert 1.55e6 < n < 1.57e6
