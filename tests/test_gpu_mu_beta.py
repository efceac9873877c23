"""The general-beta multiplicative update on the tensor-core path (beta >= 0 other than 1 and 2, rank <= 64, two planes).

One pass over X forms the model tile K = U V on chip and contracts two operand tiles against the same factor slab: the
numerator (K^(beta-2) * X) V^T and the denominator K^(beta-1) V^T (mu.py:92-97), plus the beta-divergence of the factors the
pass started from.  The finish kernel sums both partial sets, applies max(F (num / den)^gamma, 1e-12) and installs the factor.

Bounds.  The beta = 1 pass meets float64 to 3e-5 per element of its numerator and 2e-5 on its cost (test_gpu_count_data.py).
Its error is that of the model tile (bf16 hi/lo factors: about 2^-17 relative per product) entering x / k with exponent 1, plus
the hi/lo split of the operand.  Here the tile enters the numerator as k^(beta-2) and the denominator as k^(beta-1), so a relative
error e of k becomes |beta-2| e and |beta-1| e: the element bounds are 3e-5 max(1, |beta-2|) and 3e-5 max(1, |beta-1|) (every term
of the contractions is positive, so a relative bound per term bounds the sum).  The cost term k^beta h_beta(x / k) moves with
ln k as -k^beta (q - 1) near q = 1, as the KL term does; away from q = 1 the error of k^beta grows with beta and that of the
power terms with |beta-2| and |beta-1|: 2e-5 max(1, |beta-1|, |beta-2|)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BETAS = [0, 0.5, 1.5, 3, 4.2]
SHAPES = [(128, 64, 16), (1000, 500, 10), (777, 1300, 33), (2048, 4096, 64)]
X_SOURCES = ["planes", "f32"]


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _plan(X, r, source, monkeypatch):
    """A plan whose general-beta pass reads X from `source`: "planes" (hi + lo) or "f32" (the fp32 copies of X)."""
    from nn_fac import _ops as ops
    monkeypatch.setenv("NNFAC_MU_F32", "0" if source == "planes" else "1")
    return ops.NMFPlan(_dev(X)).bind_rank(r)


def _smooth(m, n, r, seed):
    rng = np.random.RandomState(seed)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    X = ((rng.rand(m, r) @ rng.rand(r, n)) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)
    return X, U, V


def _den(plan, side):
    """Sum of the denominator partials of the last pass over `side`, in split order (r x rows)."""
    info = plan.info(side)
    R = plan.m if side == 0 else plan.n
    r_pad, ld = -(-plan.r // 16) * 16, -(-R // 128) * 128
    parts = plan._den[:info["splits"] * r_pad * ld].view(info["splits"], r_pad, ld)
    out = torch.zeros((plan.r, R), dtype=torch.float32, device="cuda")
    for s in range(info["splits"]):
        out += parts[s, :plan.r, :R]
    return out


def _rtol(beta):
    return 3e-5 * max(1.0, abs(beta - 2)), 3e-5 * max(1.0, abs(beta - 1)), 2e-5 * max(1.0, abs(beta - 1), abs(beta - 2))


def _ref(X, U, V, beta):
    """float64 on the GPU: numerators and denominators of both sides."""
    X64, U64, V64 = _dev(X).double(), _dev(U).double(), _dev(V).double()
    K = U64 @ V64
    P, Q = K ** (beta - 2) * X64, K ** (beta - 1)
    return {0: (V64 @ P.T, V64 @ Q.T), 1: (U64.T @ P, U64.T @ Q)}


@pytest.mark.parametrize("x_source", X_SOURCES)
@pytest.mark.parametrize("m,n,r", SHAPES)
@pytest.mark.parametrize("beta", BETAS)
def test_beta_pass_matches_float64(beta, m, n, r, x_source, monkeypatch):
    """Numerator, denominator and cost of one pass over each side against float64; a second run of the pass gives the same
    bits; the pass without the cost gives the same partials."""
    from oracle import nnfac_oracle as orc
    X, U, V = _smooth(m, n, r, m * 7 + n + r)
    plan = _plan(X, r, x_source, monkeypatch)
    plan.set_factor(0, _dev(U.T))
    plan.set_factor(1, _dev(V))
    ref = _ref(X, U, V, beta)
    cost_ref = orc.beta_divergence(X.astype(np.float64), U.astype(np.float64) @ V.astype(np.float64), beta)
    rt_num, rt_den, rt_cost = _rtol(beta)
    for side in (0, 1):
        cost = plan.fused_beta(side, beta)
        assert (plan._xf32 is None) == (x_source == "planes")
        num, den = plan.reduce(side), _den(plan, side)
        np.testing.assert_allclose(num.double().cpu().numpy(), ref[side][0].cpu().numpy(), rtol=rt_num)
        np.testing.assert_allclose(den.double().cpu().numpy(), ref[side][1].cpu().numpy(), rtol=rt_den)
        np.testing.assert_allclose(cost.item(), cost_ref, rtol=rt_cost)
        parts, dparts = plan.reduce(side).clone(), plan._den.clone()
        cost2 = plan.fused_beta(side, beta)
        assert torch.equal(plan.reduce(side), parts) and torch.equal(plan._den, dparts) and cost2.item() == cost.item()
        assert plan.fused_beta(side, beta, want_cost=False) is None
        assert torch.equal(plan.reduce(side), parts) and torch.equal(plan._den, dparts)


@pytest.mark.parametrize("beta", [0, 0.5])
def test_beta_pass_on_count_data_with_zeros(beta, monkeypatch):
    """Poisson counts with about half of the entries exactly 0 and ragged tiles: the cost is finite and follows the oracle's
    rule for x = 0 (-1 at beta = 0, k^beta / beta above); no NaN in the partials nor in the updated factors."""
    from nn_fac.utils.beta_divergence import gamma_beta
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(11)
    m, n, r = 1100, 900, 20
    X = rng.poisson(0.7, (m, n)).astype(np.float32)
    assert 0.4 < (X == 0).mean() < 0.6
    U = (rng.rand(m, r) * 0.2 + 0.01).astype(np.float32)
    V = (rng.rand(r, n) * 0.2 + 0.01).astype(np.float32)
    plan = _plan(X, r, "f32", monkeypatch)
    plan.set_factor(0, _dev(U.T))
    plan.set_factor(1, _dev(V))
    want = orc.beta_divergence(X.astype(np.float64), U.astype(np.float64) @ V.astype(np.float64), beta)
    cost = plan.fused_beta(0, beta).item()
    assert np.isfinite(cost)
    np.testing.assert_allclose(cost, want, rtol=_rtol(beta)[2])
    assert torch.isfinite(plan.reduce(0)).all() and torch.isfinite(_den(plan, 0)).all()
    Ut = plan.mu_finish_beta(0, _dev(U.T), gamma_beta(beta), 1e-12)
    plan.fused_beta(1, beta, want_cost=False)
    assert torch.isfinite(plan.reduce(1)).all() and torch.isfinite(_den(plan, 1)).all()
    V1 = plan.mu_finish_beta(1, _dev(V), gamma_beta(beta), 1e-12)
    assert torch.isfinite(Ut).all() and torch.isfinite(V1).all() and (Ut >= 1e-12).all() and (V1 >= 1e-12).all()
    U1_ref = orc.mu_betadivmin(U.astype(np.float64), V.astype(np.float64), X.astype(np.float64), beta)
    np.testing.assert_allclose(Ut.double().cpu().numpy().T, U1_ref, rtol=2e-4)


def _data(regime, m, n, r, seed):
    rng = np.random.RandomState(seed)
    if regime == "smooth":
        X = rng.rand(m, r) @ rng.rand(r, n) + 0.1 * rng.rand(m, n)
    else:
        X = rng.poisson(3.0 * (rng.rand(m, r) @ rng.rand(r, n)) / r).astype(np.float64)
    return X.astype(np.float32), rng.rand(m, r).astype(np.float32), rng.rand(r, n).astype(np.float32)


class _NoCudaCorePath:
    def __init__(self, *a, **k):
        raise AssertionError("the CUDA-core MU path ran instead of the tensor-core pass")


@pytest.mark.parametrize("regime", ["smooth", "poisson"])
@pytest.mark.parametrize("beta", [0, 0.5, 1.5, 3])
def test_nmf_general_beta_against_oracle(beta, regime, monkeypatch):
    """nmf(update_rule="mu", beta) at 2500 x 1800, rank 20 -- above config.small_problem_elements, so float32 data takes the
    tensor-core pass under "auto" -- for 30 iterations: final objective within 1e-4 of the float64 oracle, the whole trajectory
    within 5e-4 of the oracle's (the bound of test_gpu_parity.py for transient iterates), and non-increasing wherever the
    oracle's is.  The reported cost need not decrease: at beta = 0 an entry with x = 0 counts -1 whatever k is (the reference's
    masked logarithm, beta_divergence.py:49-50), while the multiplicative update decreases the divergence in which that entry
    contributes log k -- on the Poisson counts here (48 % zeros) the oracle's own cost rises from -1.87e6 to -1.29e6."""
    import nn_fac.nmf as nmf
    from nn_fac import config
    from oracle import nnfac_oracle as orc
    m, n, r = 2500, 1800, 20
    assert m * n > config.small_problem_elements and config.precision == "auto"
    X, U0, V0 = _data(regime, m, n, r, 5)
    monkeypatch.setattr(nmf, "DeviceNMF", _NoCudaCorePath)
    U, V, costs, _ = nmf.nmf(X, r, init="custom", U_0=U0, V_0=V0, n_iter_max=30, tol=0, update_rule="mu", beta=beta,
                             return_costs=True)
    assert U.dtype == np.float32 and len(costs) == 30
    _, _, ref, _ = orc.compute_nmf(X.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64), n_iter_max=30, tol=0,
                                   update_rule="mu", beta=beta)
    assert abs(costs[-1] - ref[-1]) <= 1e-4 * abs(ref[-1]), (costs[-1], ref[-1])
    np.testing.assert_allclose(costs, ref, rtol=5e-4)
    for i in range(1, len(ref)):
        if ref[i] <= ref[i - 1]:
            assert costs[i] <= costs[i - 1] + 1e-6 * abs(costs[i - 1]), (i, costs[i - 1], costs[i])
    if beta > 0 or regime == "smooth":
        assert all(b <= a for a, b in zip(ref, ref[1:]))     # the MU property (Fevotte & Idier), where no x = 0 is masked


def test_nmf_general_beta_fixed_mode_and_tol(monkeypatch):
    """fixed_modes=[1] leaves V untouched and follows the oracle; a tol stop ends at the oracle's iteration and drops the
    speculative iteration (the returned factors are the ones the last reported cost belongs to)."""
    import nn_fac.nmf as nmf
    from oracle import nnfac_oracle as orc
    m, n, r, beta = 2500, 1800, 20, 0.5
    X, U0, V0 = _data("smooth", m, n, r, 9)
    X64, U64, V64 = X.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64)
    monkeypatch.setattr(nmf, "DeviceNMF", _NoCudaCorePath)
    U, V, costs, _ = nmf.nmf(X, r, init="custom", U_0=U0, V_0=V0, n_iter_max=8, tol=0, update_rule="mu", beta=beta,
                             fixed_modes=[1], return_costs=True)
    _, _, ref, _ = orc.compute_nmf(X64, U64, V64, n_iter_max=8, tol=0, update_rule="mu", beta=beta, fixed_modes=[1])
    assert np.array_equal(V, V0)
    assert abs(costs[-1] - ref[-1]) <= 1e-4 * ref[-1]
    _, _, full, _ = orc.compute_nmf(X64, U64, V64, n_iter_max=40, tol=0, update_rule="mu", beta=beta)
    steps = np.abs(np.diff(full))
    tol = float(np.sqrt(steps[14] * steps[15]))          # between two consecutive steps: the stop falls at iteration 16
    U, V, costs, _ = nmf.nmf(X, r, init="custom", U_0=U0, V_0=V0, n_iter_max=40, tol=tol, update_rule="mu", beta=beta,
                             return_costs=True)
    assert len(costs) == 17, len(costs)
    K = U.astype(np.float64) @ V.astype(np.float64)
    assert abs(orc.beta_divergence(X64, K, beta) - costs[-1]) <= 1e-4 * costs[-1]


def _f64_beta_chunked(X, Ut, V, beta, rows=4096):
    from oracle import nnfac_oracle as orc
    tot = 0.0
    V64 = V.double()
    for lo in range(0, X.shape[0], rows):
        x = X[lo:lo + rows].double()
        k = Ut[:, lo:lo + rows].double().T @ V64
        if beta == 0:
            q = x / k
            tot += float((q - torch.where(x != 0, torch.log(q), torch.zeros_like(q)) - 1).sum())
        else:
            tot += orc.beta_divergence(x.cpu().numpy(), k.cpu().numpy(), beta)
    return tot


def test_nmf_config2_full_size_beta0_against_oracle_on_subsamples():
    """C2 (65536 x 8192, rank 64) with Itakura-Saito: the reported objective against a float64 evaluation over the whole matrix;
    one outer iteration against the oracle on random rows of U and columns of V (an MU update couples no rows)."""
    from nn_fac import _fast
    from oracle import nnfac_oracle as orc
    m, n, r, beta = 65536, 8192, 64, 0
    g = torch.Generator(device="cuda"); g.manual_seed(2024)
    W0, H0 = torch.rand((m, r), generator=g, device="cuda"), torch.rand((r, n), generator=g, device="cuda")
    X = W0 @ H0
    X += float(X.mean()) * torch.rand((m, n), generator=g, device="cuda") + 1e-3
    del W0, H0
    U0, V0 = torch.rand((m, r), generator=g, device="cuda"), torch.rand((r, n), generator=g, device="cuda")
    assert _fast.eligible(torch.float32, r, "mu", beta)
    st = _fast.FusedNMF(X, U0, V0)
    costs, _ = st.run(3, 0.0, "mu", beta=beta)
    assert len(costs) == 3 and costs[0] >= costs[1] >= costs[2] > 0
    want = _f64_beta_chunked(X, st.Ut, st.V, beta)
    assert abs(costs[-1] - want) <= 1e-5 * want, (costs[-1], want)

    st = _fast.FusedNMF(X, U0, V0)
    st.run(1, 0.0, "mu", beta=beta)
    U1t, V1 = st.Ut, st.V
    rs = np.random.RandomState(5)
    rows = torch.from_numpy(np.sort(rs.choice(m, 192, replace=False))).cuda()
    cols = torch.from_numpy(np.sort(rs.choice(n, 192, replace=False))).cuda()
    Xr, Xc = X[rows].double().cpu().numpy(), X[:, cols].double().cpu().numpy()
    U0r, V0c = U0[rows].double().cpu().numpy(), V0[:, cols].double().cpu().numpy()
    V0h, U1h = V0.double().cpu().numpy(), U1t.double().cpu().numpy().T
    want_U = orc.mu_betadivmin(U0r, V0h, Xr, beta)                                   # mu.py:92-97
    want_V = orc.mu_betadivmin(V0c.T, U1h.T, Xc.T, beta).T                           # mu.py:27
    got_U, got_V = U1h[rows.cpu().numpy()], V1[:, cols].double().cpu().numpy()
    assert np.linalg.norm(got_U - want_U) <= 2e-4 * np.linalg.norm(want_U)
    assert np.linalg.norm(got_V - want_V) <= 2e-4 * np.linalg.norm(want_V)
    assert (got_U >= 0).all() and (got_V >= 0).all()
