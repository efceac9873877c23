"""CPU checks of the "fp32x3" precision mode: the setting, its routing rules and the C ABI entry points of 3-plane plans."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.test_abi import HEADER, LIB, declared_symbols

NEW_SYMBOLS = ("nnfac_nmf_plan_bytes_planes", "nnfac_nmf_plan_create_planes")


@pytest.fixture(autouse=True)
def _restore_precision():
    from nn_fac import config
    yield
    config.set_precision("auto")


def test_fp32x3_is_accepted_and_bad_names_still_raise():
    from nn_fac import config
    config.set_precision("fp32x3")
    assert config.precision == "fp32x3"
    with pytest.raises(ValueError):
        config.set_precision("fp24")
    assert config.precision == "fp32x3"


@pytest.mark.parametrize("numel", [10, 1 << 22, (1 << 22) + 1, 1 << 30])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_working_dtype_under_fp32x3(numel, dtype):
    from nn_fac import _lib as L
    from nn_fac import config
    config.set_precision("fp32x3")
    a = np.zeros((2, 2), dtype=dtype)
    assert L.working_dtype(numel, a, a, a) == (torch.float64, torch.float32)
    assert L.resolve_dtype(a) == torch.float64        # direct calls of the update rules compute in float64


def test_working_dtype_of_the_other_modes_is_unchanged():
    from nn_fac import _lib as L
    from nn_fac import config
    a32, a64 = np.zeros(1, np.float32), np.zeros(1, np.float64)
    assert L.working_dtype(10, a32) == (torch.float64, torch.float32)
    assert L.working_dtype(1 << 23, a32) == (torch.float32, torch.float32)
    assert L.working_dtype(1 << 23, a64) == (torch.float64, torch.float64)
    config.set_precision("fp32")
    assert L.working_dtype(10, a64) == (torch.float32, torch.float32)
    config.set_precision("fp64")
    assert L.working_dtype(1 << 23, a32) == (torch.float64, torch.float64)


def test_eligible_with_three_planes():
    from nn_fac import _fast
    for rank in (1, 16, 33, 64, 65, 96, 128, 129):
        for rule, beta in (("hals", 2), ("mu", 1), ("mu", 2), ("mu", 0), ("mu", 0.5), ("mu", 3)):
            expect = rank <= 64 and (rule == "hals" or beta in (1, 2))
            assert _fast.eligible(torch.float32, rank, rule, beta, planes=3) == expect, (rank, rule, beta)
        assert not _fast.eligible(torch.float64, rank, "hals", 2, planes=3)
    # two planes: as before
    assert _fast.eligible(torch.float32, 128, "hals", 2) and not _fast.eligible(torch.float32, 65, "mu", 1)


def test_planes_follow_the_precision():
    from nn_fac import _fast, config
    assert _fast.planes_of_precision() == 2
    config.set_precision("fp32x3")
    assert _fast.planes_of_precision() == 3
    config.set_precision("fp32")
    assert _fast.planes_of_precision() == 2


def test_sharded_refuses_fp32x3_before_any_device_work():
    from nn_fac import config, sharded
    config.set_precision("fp32x3")
    rng = np.random.RandomState(0)
    with pytest.raises(NotImplementedError):
        sharded.compute_nmf_sharded(rng.rand(8, 6).astype(np.float32), 2, rng.rand(8, 2).astype(np.float32),
                                    rng.rand(2, 6).astype(np.float32), n_iter_max=1)


def test_plane_count_abi_is_declared_bound_and_exported():
    from nn_fac import _lib
    syms = declared_symbols()
    text = open(HEADER).read()
    assert "NNFAC_HALS_NO_TC" in text
    for name in NEW_SYMBOLS:
        assert name in syms
        assert name in _lib.SIGNATURES
    assert os.path.exists(LIB), "build the library first: bash nn-fac_b200/build.sh"
    lib = ctypes.CDLL(LIB)
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name)
    assert _lib.HALS_NO_TC == 4


def test_results_are_cast_to_float32_only_under_fp32x3():
    from nn_fac import _lib as L
    from nn_fac import config
    a64, t64 = np.ones((2, 3)), torch.ones((2, 3), dtype=torch.float64)
    assert L.as_output(a64) is a64 and L.as_output(t64) is t64
    config.set_precision("fp32x3")
    assert L.as_output(a64).dtype == np.float32 and L.as_output(t64).dtype == torch.float32
    np.testing.assert_array_equal(L.as_output(a64), a64)
