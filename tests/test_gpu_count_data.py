"""The beta = 1 fused pass on both of its X sources, and the fp32 tensor-core path on count data with exact zeros.

The beta = 1 pass reads X either from fp32 copies of the planes (made on first use when memory allows) or rebuilds x = hi + lo
from the bf16 planes (what runs when X is too large for the copies).  NNFAC_MU_F32=0 / 1 forces one or the other on a fresh plan.
Count data (KL-NMF's usual input) has exact zeros, whole zero rows and columns: x = 0 takes dedicated code in the fused pass
(0 * log of the ratio, k g(0) = k in the 3-plane pass) and drives rows of the factors to the floor."""
import functools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

X_SOURCES = ["planes", "f32"]


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _plan(X, r, source, monkeypatch):
    """A plan whose beta = 1 pass reads X from `source`: "planes" (hi + lo), "f32" (the fp32 copies) or "3planes" (a 3-plane plan,
    whose beta = 1 pass always reads its fp32 copies)."""
    from nn_fac import _ops as ops
    monkeypatch.setenv("NNFAC_MU_F32", "0" if source == "planes" else "1")
    plan = ops.NMFPlan(_dev(X)).bind_rank(r, planes=3 if source == "3planes" else 2)
    if source != "planes":
        plan.enable_f32()
    return plan


def _check_source(plan, source):
    """The pass ran on the X source the test asked for."""
    assert (plan._xf32 is None) == (source == "planes"), source


def _smooth(m, n, r, seed):
    """The data of test_gpu_tc.py::test_fused_pass_matches_float64 (positive, no zeros)."""
    rng = np.random.RandomState(seed)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    X = ((rng.rand(m, r) @ rng.rand(r, n)) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)
    return X, U, V


SHAPES = [(128, 64, 16), (384, 320, 64), (1000, 500, 10), (777, 1300, 33), (2048, 4096, 64), (100, 3000, 16)]


# ---------------------------------------------------------------------------------------------
# A. X source of the beta = 1 pass
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("x_source", X_SOURCES)
@pytest.mark.parametrize("m,n,r", SHAPES)
def test_beta1_pass_matches_float64_on_either_x_source(m, n, r, x_source, monkeypatch):
    """Numerators and KL(X | UV) of the beta = 1 pass against float64 numpy, both sides, with and without the cost (COST is a
    template flag: both instantiations); the numerator does not depend on whether the cost was wanted."""
    X, U, V = _smooth(m, n, r, m * 7 + n + r)
    plan = _plan(X, r, x_source, monkeypatch)
    plan.set_factor(0, _dev(U.T))
    plan.set_factor(1, _dev(V))
    X64, U64, V64 = X.astype(np.float64), U.astype(np.float64), V.astype(np.float64)
    K = U64 @ V64
    kl = np.sum(X64 * np.log(X64 / K) - X64 + K)
    for side, ref in ((0, V64 @ (X64 / K).T), (1, U64.T @ (X64 / K))):
        out, cost = plan.fused(side, 1)
        _check_source(plan, x_source)
        np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=3e-5)
        np.testing.assert_allclose(cost.item(), kl, rtol=2e-5)
        out_nc, cost_nc = plan.fused(side, 1, want_cost=False)
        assert cost_nc is None
        assert torch.equal(out_nc, out)


@pytest.mark.parametrize("m,n,r", SHAPES)
def test_beta1_pass_planes_and_f32_copies_are_bit_identical(m, n, r, monkeypatch):
    """x = hi + lo is the same fp32 value whether the pass adds the planes or reads the copy made from them: same bits."""
    X, U, V = _smooth(m, n, r, m * 7 + n + r)
    res = {}
    for source in X_SOURCES:
        plan = _plan(X, r, source, monkeypatch)
        plan.set_factor(0, _dev(U.T))
        plan.set_factor(1, _dev(V))
        res[source] = [plan.fused(side, 1) for side in (0, 1)] + [plan.fused(side, 1, want_cost=False)[0] for side in (0, 1)]
        _check_source(plan, source)
    a, b = res["planes"], res["f32"]
    for side in (0, 1):
        assert torch.equal(a[side][0], b[side][0]) and torch.equal(a[side][1], b[side][1]), side
        assert torch.equal(a[2 + side], b[2 + side]) and torch.equal(a[2 + side], a[side][0]), side


def test_fused_nmf_mu_beta1_is_bit_identical_on_either_x_source(monkeypatch):
    """Five MU iterations (beta = 1) of the fused driver: the X source changes no bit of the costs or the factors; the objective
    follows the float64 oracle."""
    from nn_fac import _fast
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(3)
    m, n, r = 3000, 2000, 32
    X = (rng.rand(m, r) @ rng.rand(r, n) + 0.3 * rng.rand(m, n)).astype(np.float32)
    U0, V0 = rng.rand(m, r).astype(np.float32), rng.rand(r, n).astype(np.float32)
    _, _, ref, _ = orc.compute_nmf(X.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64), n_iter_max=5, tol=0,
                                   update_rule="mu", beta=1)
    assert _fast.eligible(torch.float32, r, "mu", 1)
    out = {}
    for source in X_SOURCES:
        monkeypatch.setenv("NNFAC_MU_F32", "0" if source == "planes" else "1")
        st = _fast.FusedNMF(X, U0, V0)
        costs, _ = st.run(5, 0.0, "mu", beta=1)
        _check_source(st.eng.plan, source)
        out[source] = (costs, st.Ut.clone(), st.V.clone())
        assert abs(costs[-1] - ref[-1]) <= 1e-4 * ref[-1], (source, costs[-1], ref[-1])
    a, b = out["planes"], out["f32"]
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


# ---------------------------------------------------------------------------------------------
# B. count data with exact zeros
# ---------------------------------------------------------------------------------------------
def _counts(m, n, mean, seed):
    """Seeded Poisson counts with whole zero rows (first, middle, last) and zero columns.  Returns X, zero rows, zero cols."""
    rng = np.random.RandomState(seed)
    X = rng.poisson(mean, size=(m, n)).astype(np.float32)
    zr, zc = [0, m // 2, m - 1], [0, n // 3, n - 1]
    X[zr, :] = 0.0
    X[:, zc] = 0.0
    return X, zr, zc


def _kl_masked(X64, K):
    """The reference's KL with its `where=` mask (beta_divergence.py:45-48): an entry x = 0 contributes k."""
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(X64 > 0, X64 * np.log(X64 / K), 0.0)
    return float(np.sum(t - X64 + K))


COUNT_CASES = [(0.5, 1000, 1300, 20), (0.05, 1000, 1300, 20), (0.5, 300, 2111, 64), (0.05, 300, 2111, 64)]


@pytest.mark.parametrize("source", ["planes", "f32", "3planes"])
@pytest.mark.parametrize("mean,m,n,r", COUNT_CASES)
def test_fused_passes_on_count_data_match_float64(mean, m, n, r, source, monkeypatch):
    """Both fused passes on Poisson data (~60 % or ~95 % exact zeros, zero rows and columns) against float64: cross products,
    ||X - UV||^2, beta = 1 numerators and the masked KL; numerator columns of zero rows / columns of X are exactly 0."""
    X, zr, zc = _counts(m, n, mean, int(mean * 100) + m + r)
    assert (X == 0).mean() > (0.55 if mean == 0.5 else 0.9)
    rng = np.random.RandomState(m + n)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    plan = _plan(X, r, source, monkeypatch)
    plan.set_factor(0, _dev(U.T))
    plan.set_factor(1, _dev(V))
    X64, U64, V64 = X.astype(np.float64), U.astype(np.float64), V.astype(np.float64)
    K = U64 @ V64
    fro = np.sum((X64 - K) ** 2)
    kl = _kl_masked(X64, K)
    Q = X64 / K
    for side, cross_ref, num_ref, zero in ((0, V64 @ X64.T, V64 @ Q.T, zr), (1, U64.T @ X64, U64.T @ Q, zc)):
        out, cost = plan.fused(side, 0)
        np.testing.assert_allclose(out.cpu().numpy(), cross_ref, rtol=2e-5)
        np.testing.assert_allclose(cost.item(), fro, rtol=2e-5)
        out, cost = plan.fused(side, 1)
        _check_source(plan, "planes" if source == "planes" else "f32")
        num = out.cpu().numpy()
        assert np.isfinite(cost.item()), (side, cost.item())
        np.testing.assert_allclose(num, num_ref, rtol=3e-5)
        np.testing.assert_allclose(cost.item(), kl, rtol=2e-5)
        assert (num[:, zero] == 0).all(), side


@pytest.mark.parametrize("x_source", X_SOURCES)
def test_mu_finish_on_zero_rows_gives_the_floor(x_source, monkeypatch):
    """A factor row whose numerator is 0 (a zero row / column of X) becomes exactly fp32(1e-12) (mu.py:88); the other rows follow
    float64."""
    from nn_fac import _ops as ops
    m, n, r = 1000, 1300, 20
    X, zr, zc = _counts(m, n, 0.5, 17)
    rng = np.random.RandomState(18)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    plan = _plan(X, r, x_source, monkeypatch)
    Ut_d, V_d = _dev(U.T), _dev(V)
    plan.set_factor(0, Ut_d)
    plan.set_factor(1, V_d)
    X64, U64, V64 = X.astype(np.float64), U.astype(np.float64), V.astype(np.float64)
    Q = X64 / (U64 @ V64)
    floor = np.float32(1e-12)
    # U first (mu.py:84-88 with the row sums of V), then V from the new U, as the driver does
    plan.fused(0, 1, want_cost=False, keep_partials=True)
    _check_source(plan, x_source)
    newUt = plan.mu_finish(0, Ut_d, ops.row_sums(V_d), 1e-12).cpu().numpy()
    assert (newUt[:, zr] == floor).all()
    want = np.maximum(U64.T * (V64 @ Q.T) / V64.sum(axis=1)[:, None], 1e-12)
    np.testing.assert_allclose(newUt, want, rtol=3e-5)
    newUt_d = _dev(newUt)
    plan.fused(1, 1, want_cost=False, keep_partials=True)
    newV = plan.mu_finish(1, V_d, ops.row_sums(newUt_d), 1e-12).cpu().numpy()
    assert (newV[:, zc] == floor).all()
    U1 = newUt.astype(np.float64).T
    want = np.maximum(V64 * (U1.T @ (X64 / (U1 @ V64))) / U1.sum(axis=0)[:, None], 1e-12)
    np.testing.assert_allclose(newV, want, rtol=3e-5)


@functools.lru_cache(maxsize=None)
def _count_problem(mean):
    m, n, r = 2500, 1800, 20                      # 4.5e6 elements > 2^22: "auto" keeps float32 data on the tensor-core path
    X, _, _ = _counts(m, n, mean, 23 if mean == 0.5 else 29)
    rng = np.random.RandomState(31)
    U0 = (rng.rand(m, r) + 0.1).astype(np.float32)
    V0 = (rng.rand(r, n) + 0.1).astype(np.float32)
    return X, U0, V0, r


@functools.lru_cache(maxsize=None)
def _count_oracle(mean, rule):
    from oracle import nnfac_oracle as orc
    X, U0, V0, r = _count_problem(mean)
    stats = {}
    beta = 1 if rule == "mu" else 2
    _, _, ref, _ = orc.compute_nmf(X.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64), n_iter_max=20, tol=0,
                                   update_rule=rule, beta=beta, stats=stats)
    return np.asarray(ref), stats


@pytest.mark.parametrize("variant", ["mu_auto", "mu_planes", "mu_fp32x3", "hals"])
@pytest.mark.parametrize("mean", [0.5, 0.05])
def test_nmf_on_count_data_tensor_core_path_vs_oracle(mean, variant, monkeypatch):
    """20 iterations of the fused driver on count data against the float64 oracle: objective within 1e-4, finite costs and
    factors, MU non-increasing, HALS sweep counts within one of the oracle's."""
    import nn_fac.config as config
    from nn_fac import _fast
    X, U0, V0, r = _count_problem(mean)
    rule = "hals" if variant == "hals" else "mu"
    beta = 2 if rule == "hals" else 1
    ref, stats = _count_oracle(mean, rule)
    if variant == "mu_planes":
        monkeypatch.setenv("NNFAC_MU_F32", "0")
    if variant == "mu_fp32x3":
        config.set_precision("fp32x3")
    try:
        assert X.size > config.small_problem_elements
        planes = _fast.planes_of_precision()
        assert planes == (3 if variant == "mu_fp32x3" else 2)
        assert _fast.eligible(torch.float32, r, rule, beta, planes=planes)
        st = _fast.FusedNMF(X, U0, V0)
        costs, _ = st.run(20, 0.0, rule, beta=beta)
        Ut, V = st.Ut.cpu().numpy(), st.V.cpu().numpy()
        sweeps = np.array([t.cpu().numpy() for t in st.sweep_log]) if rule == "hals" else None
        if variant == "mu_planes":
            assert st.eng.plan._xf32 is None
        elif rule == "mu":
            assert st.eng.plan._xf32 is not None
    finally:
        config.set_precision("auto")
    costs = np.asarray(costs)
    assert len(costs) == 20 and np.isfinite(costs).all(), costs
    assert not np.isnan(Ut).any() and not np.isnan(V).any()
    assert abs(costs[-1] - ref[-1]) <= 1e-4 * ref[-1], (costs[-1], ref[-1])
    if rule == "mu":
        assert np.all(np.diff(costs) <= 1e-9 * costs[0]), np.diff(costs)
    else:
        want = np.stack([stats["sweeps_U"], stats["sweeps_V"]], axis=1)
        assert np.abs(sweeps - want).max() <= 1, (sweeps, want)
