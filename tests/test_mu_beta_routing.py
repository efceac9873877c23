"""CPU checks of the general-beta MU pass: which problems the tensor-core path takes, the sharded path's refusal before any
device work, and the C ABI entry points (declared, bound, exported)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.test_abi import LIB, declared_symbols

NEW_SYMBOLS = ("nnfac_nmf_plan_fused_beta_bytes", "nnfac_nmf_plan_fused_beta", "nnfac_nmf_plan_mu_finish_beta")


def test_eligible_routes_every_beta_at_rank_64_and_below():
    from nn_fac import _fast
    for rank in (1, 16, 33, 64, 65, 128):
        for beta in (0, 0.25, 0.5, 1, 1.5, 2, 3, 4.2, 7):
            expect = rank <= 64 or (beta == 2 and rank <= 128)
            assert _fast.eligible(torch.float32, rank, "mu", beta) == expect, (rank, beta)
            assert not _fast.eligible(torch.float64, rank, "mu", beta)
        assert not _fast.eligible(torch.float32, rank, "mu", -0.5)
    assert _fast.eligible(torch.float32, 128, "hals", 2) and not _fast.eligible(torch.float32, 129, "hals", 2)


def test_eligible_with_three_planes_is_unchanged():
    from nn_fac import _fast
    for beta in (0, 0.5, 1.5, 3):
        assert not _fast.eligible(torch.float32, 16, "mu", beta, planes=3)
    assert _fast.eligible(torch.float32, 64, "mu", 1, planes=3) and _fast.eligible(torch.float32, 64, "mu", 2, planes=3)


def test_general_beta_selects_both_contractions():
    from nn_fac import _fast
    assert [b for b in (0, 0.5, 1, 1.5, 2, 3) if _fast.general_beta("mu", b)] == [0, 0.5, 1.5, 3]
    assert not _fast.general_beta("hals", 2)


@pytest.mark.parametrize("beta", [0, 3])
def test_sharded_refuses_general_beta_before_any_device_work(beta):
    from nn_fac import sharded
    rng = np.random.RandomState(0)
    with pytest.raises(NotImplementedError):
        sharded.compute_nmf_sharded(rng.rand(8, 6).astype(np.float32), 2, rng.rand(8, 2).astype(np.float32),
                                    rng.rand(2, 6).astype(np.float32), n_iter_max=1, update_rule="mu", beta=beta)


def test_fused_nmf_refuses_general_beta_over_several_ranks():
    from nn_fac import _fast
    st = _fast.FusedNMF.__new__(_fast.FusedNMF)
    st.comm = _fast.Comm()
    st.comm.world = 2
    with pytest.raises(NotImplementedError):
        st.run(1, 0.0, "mu", beta=0)


def test_new_entry_points_are_declared_bound_and_exported():
    from nn_fac import _lib
    syms = declared_symbols()
    for name in NEW_SYMBOLS:
        assert name in syms and name in _lib.SIGNATURES
    assert os.path.exists(LIB), "build the library first: bash nn-fac_b200/build.sh"
    lib = ctypes.CDLL(LIB)
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name)
