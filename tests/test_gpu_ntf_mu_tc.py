"""The NTF multiplicative update on the tensor core (3-way fp32 tensors, rank <= 64, every beta >= 0) against float64.

The MU / general-beta pass of tc_fused_kernel on the plans DeviceNTF builds -- mode 0's one-sided plan, middle-mode views
(3-D map) and last-mode views (MN-major tile read transposed) -- with the Khatri-Rao operand of set_krao: its numerator and
denominator partials and its cost element-wise against a float64 evaluation of the same operands; then whole ntf() runs against
the float64 oracle, the memory they take, and the routes that keep the CUDA-core update.
"""
import numpy as np
import pytest

from tests.test_gpu_ntf_tc import MTTKRP_SHAPES, _dev, _kind, _krao_t, _ntf_problem, _state, _strided

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _tensor_core_path(fp32_path):
    """Everything in this file is about the float32 kernels, whatever the size of the problem."""
    yield


# ---------------------------------------------------------------------------------------------
# 1. One pass against float64
# ---------------------------------------------------------------------------------------------
PASS_SHAPES = [s for s in MTTKRP_SHAPES if len(s) == 3]     # I = 5, 8, 72, 130, 200 and two row tiles of mode 0


def _pass(plan, Ft, At, Bt, beta):
    """set_factor_rows(F^T) + set_krao(At, Bt) + the MU pass with cost; returns (numerator, denominator or None, cost) on the host
    (denominator: the sum of the partials in the order of the reduction)."""
    import torch
    plan.set_factor_rows(_dev(Ft))
    plan.set_krao(_strided(At), _strided(Bt))
    if beta == 1:
        num, cost = plan.fused(0, 1, want_cost=True)
        return num.cpu().numpy(), None, float(cost.item())
    cost = plan.fused_beta(0, beta, want_cost=True)
    num = plan.reduce(0)
    info = plan.info(0)
    ldp = -(-plan.m // 128) * 128
    den = plan._den[:info["splits"] * ((plan.r + 15) // 16 * 16) * ldp].reshape(info["splits"], -1, ldp)
    den_sum = torch.zeros((plan.r, plan.m), dtype=torch.float32, device="cuda")
    for s in range(info["splits"]):
        den_sum += den[s, :plan.r, :plan.m]
    return num.cpu().numpy(), den_sum.cpu().numpy(), float(cost.item())


def _reference(T64, mode, F64, Kt64, beta):
    """float64 numerator (K^(beta-2) X) krao, denominator K^(beta-1) krao (both r x I) and d_beta(X | K), K = F krao^T."""
    from oracle import nnfac_oracle as orc
    X = orc.unfold(T64, mode)
    K = F64 @ Kt64
    num = ((K ** (beta - 2.0)) * X) @ Kt64.T
    den = (K ** (beta - 1.0)) @ Kt64.T
    return num.T, den.T, orc.beta_divergence(X, K, beta), K


# Bounds.  Each operand carries two bf16 planes (2^-17 relative), the model tile adds the dropped lo * lo term and the truncating
# fp32 accumulation (together <= ~3e-5 relative on positive data), the ratio tiles K^(beta-2) X and K^(beta-1) inherit |beta - 2|
# resp. |beta - 1| times that, and the contraction adds another ~3e-5: 1e-4 (1 + |beta - 2|) relative, element by element (all
# terms are positive).  The cost: 1e-4 of sum k^beta |x / k - 1| (the model error times the derivative of the terms), 1e-6 of the
# size of the terms (MUFU.LG2 / EX2 and fp32 partial sums), plus 1e-6 of sum x for beta = 1, whose cost is sum x ln(x / k)
# - sum x + sum k.
def _bounds(num64, den64, T64, K, mode, beta):
    from oracle import nnfac_oracle as orc
    X = orc.unfold(T64, mode)
    rel = 1e-4 * (1.0 + abs(beta - 2.0))
    kb = K ** beta
    cbound = 1e-4 * float((kb * np.abs(X / K - 1.0)).sum()) + 1e-6 * float(kb.sum() + (X ** beta).sum())
    if beta == 1:
        cbound += 1e-6 * float(X.sum())
    return rel * num64, rel * den64, cbound


@pytest.mark.parametrize("beta", [1, 0, 0.5, 3])
@pytest.mark.parametrize("r", [5, 33, 64])
@pytest.mark.parametrize("shape", PASS_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_mu_pass_of_every_mode_matches_float64(shape, r, beta, monkeypatch):
    """The pass on the plan of each mode (full, middle view, last view) against float64, element-wise; each view gives the same
    bits as the copy plan of the same unfolding (NNFAC_NTF_VIEWS=0), and a second run the same bits as the first."""
    rng = np.random.RandomState(sum(shape) + 10 * r + int(10 * beta))
    T = (rng.rand(*shape) + 0.1).astype(np.float32)
    Fs = [(rng.rand(s, r) + 0.1).astype(np.float32) for s in shape]
    views, copies = _state(T, r, monkeypatch), _state(T, r, monkeypatch, views=False)
    assert " ".join(_kind(p) for p in views.plans) == MTTKRP_SHAPES[shape]
    T64 = T.astype(np.float64)
    worst = 0.0
    for mode in range(3):
        a, b = (i for i in range(3) if i != mode)
        Ft, At, Bt = np.ascontiguousarray(Fs[mode].T), np.ascontiguousarray(Fs[a].T), np.ascontiguousarray(Fs[b].T)
        got = _pass(views.plans[mode], Ft, At, Bt, beta)
        again = _pass(views.plans[mode], Ft, At, Bt, beta)
        copy = _pass(copies.plans[mode], Ft, At, Bt, beta)
        Kt64 = _krao_t(At.astype(np.float64), Bt.astype(np.float64))
        num64, den64, cost64, K = _reference(T64, mode, Fs[mode].astype(np.float64), Kt64, beta)
        nb, db, cb = _bounds(num64, den64, T64, K, mode, beta)
        err = np.abs(got[0] - num64)
        assert (err <= nb).all(), (mode, "numerator", float((err / nb).max()))
        worst = max(worst, float((err / nb).max()))
        if beta != 1:
            err = np.abs(got[1] - den64)
            assert (err <= db).all(), (mode, "denominator", float((err / db).max()))
        assert abs(got[2] - cost64) <= cb, (mode, got[2], cost64, cb)
        for other in (again, copy):
            np.testing.assert_array_equal(got[0], other[0])
            if beta != 1:
                np.testing.assert_array_equal(got[1], other[1])
        assert got[2] == again[2]
        if beta != 1:
            assert got[2] == copy[2]
        else:   # the cost adds the sum of X, which each plan forms over its own layout (fp32 sums of 16 elements, then fp64)
            assert abs(got[2] - copy[2]) <= 1e-6 * float(T64.sum()), (mode, got[2], copy[2])
    print(f"{shape} r={r} beta={beta}: worst numerator error / bound = {worst:.3g}")


@pytest.mark.parametrize("beta", [0, 1])
def test_mu_pass_on_count_data_follows_the_masked_rule(beta, monkeypatch):
    """Count data with exact zeros (a third of the entries): the cost is finite and equals the reference's masked rule (x = 0
    contributes k for beta = 1, -1 for beta = 0) within the bound of section 1, on every plan kind."""
    shape, r = (64, 96, 72), 8
    rng = np.random.RandomState(7 + beta)
    T = rng.poisson(1.0, size=shape).astype(np.float32)
    assert (T == 0).mean() > 0.3
    Fs = [(rng.rand(s, r) + 0.1).astype(np.float32) for s in shape]
    state = _state(T, r, monkeypatch)
    T64 = T.astype(np.float64)
    for mode in range(3):
        a, b = (i for i in range(3) if i != mode)
        Ft, At, Bt = np.ascontiguousarray(Fs[mode].T), np.ascontiguousarray(Fs[a].T), np.ascontiguousarray(Fs[b].T)
        num, _, cost = _pass(state.plans[mode], Ft, At, Bt, beta)
        Kt64 = _krao_t(At.astype(np.float64), Bt.astype(np.float64))
        _, _, cost64, K = _reference(T64, mode, Fs[mode].astype(np.float64), Kt64, beta)
        _, _, cb = _bounds(np.zeros(1), np.zeros(1), T64, K, mode, beta)
        assert np.isfinite(cost) and np.isfinite(num).all()
        assert abs(cost - cost64) <= cb, (mode, cost, cost64, cb)


# ---------------------------------------------------------------------------------------------
# 2. Whole runs against the float64 oracle
# ---------------------------------------------------------------------------------------------
SHAPE, RANK = (256, 128, 192), 16     # modes 1 and 2 are views (right = 192 is a multiple of 64; last I = 192)


def _run(T, F0, kw, n_iter_max=10, tol=-1, beta=1):
    import nn_fac.ntf as ntf
    args = dict(sparsity_coefficients=[None] * 3, fixed_modes=[], normalize=[False] * 3)
    args.update({k: list(v) for k, v in kw.items()})
    return ntf.ntf(T, RANK, init="custom", factors_0=[f.copy() for f in F0], n_iter_max=n_iter_max, tol=tol, return_costs=True,
                   update_rule="mu", beta=beta, **args)


def _oracle(T, F0, kw, beta, n_iter_max=10):
    from oracle import nnfac_oracle as orc
    args = {k: list(v) for k, v in kw.items()}
    return orc.compute_ntf(T.astype(np.float64), RANK, [f.astype(np.float64) for f in F0], n_iter_max=n_iter_max, tol=-1,
                           update_rule="mu", beta=beta, **args)[1]


def _count_model(monkeypatch):
    """Counts the tensor-sized models the old path forms (DeviceNTF.reconstruct_unfolded)."""
    import nn_fac.ntf as ntf
    calls = []
    orig = ntf.DeviceNTF.reconstruct_unfolded
    monkeypatch.setattr(ntf.DeviceNTF, "reconstruct_unfolded", lambda self, *a: calls.append(1) or orig(self, *a))
    return calls


RUN_CASES = {
    "beta1": (1, {}),
    "beta2": (2, {}),
    "beta0": (0, {}),
    "beta1.5": (1.5, {}),
    "beta1-fixed0": (1, dict(fixed_modes=[0])),
    "beta0-fixed1": (0, dict(fixed_modes=[1])),
    "beta2-fixed0": (2, dict(fixed_modes=[0])),
    "beta1.5-sparsity": (1.5, dict(sparsity_coefficients=[0.05, None, 0.02])),
}


@pytest.mark.parametrize("case", list(RUN_CASES))
def test_ntf_mu_runs_match_float64(case, monkeypatch):
    """10 iterations of ntf(update_rule="mu") from fp32 inputs on the tensor core against the float64 oracle: the objective within
    1e-4 relative at every iteration, no tensor-sized model formed; with a copy for every mode (NNFAC_NTF_VIEWS=0) the same
    factors bit for bit."""
    beta, kw = RUN_CASES[case]
    T, F0 = _ntf_problem(SHAPE, RANK, 0.4, seed=11)
    state = _state(T, RANK, monkeypatch)
    assert " ".join(_kind(p) for p in state.plans) == "full view view" and state.direct_cost("mu", kw.get("fixed_modes", ()))
    del state
    ref = _oracle(T, F0, kw, beta)
    calls = _count_model(monkeypatch)
    fa, costs, _ = _run(T, F0, kw, beta=beta)
    assert not calls
    np.testing.assert_allclose(costs, ref, rtol=1e-4)
    print(f"{case}: worst relative objective error {float(np.max(np.abs(np.array(costs) / ref - 1))):.3g}")
    monkeypatch.setenv("NNFAC_NTF_VIEWS", "0")
    fb, copies, _ = _run(T, F0, kw, beta=beta)
    for a, b in zip(fa, fb):
        np.testing.assert_array_equal(a, b)
    # the cost pass of a view and of a copy sum the same terms; beta = 2 with mode 0 fixed: over unfold(T, 0) and over the copy
    # of unfold(T, 1), the same quantity in another order
    np.testing.assert_allclose(copies, costs, rtol=2e-5)


@pytest.mark.parametrize("beta", [1, 0])
def test_ntf_mu_tol_stop_rolls_back_two_iterations(beta):
    """A tol stop returns the uncut run's costs cut at the same place and the factors of the same iterations run without a stop,
    with graph replay (12 iterations) and without (short runs launch eagerly)."""
    T, F0 = _ntf_problem(SHAPE, RANK, 0.4, seed=12)
    _, full, _ = _run(T, F0, {}, n_iter_max=12, beta=beta)
    tol = 0.5 * (abs(full[5] - full[6]) + abs(full[6] - full[7]))
    stop = next(k for k in range(1, 12) if abs(full[k - 1] - full[k]) < tol)
    assert stop < 11
    fa, ca, _ = _run(T, F0, {}, n_iter_max=12, tol=tol, beta=beta)
    assert len(ca) == stop + 1
    np.testing.assert_allclose(ca, full[:stop + 1], rtol=1e-6)
    fb, _, _ = _run(T, F0, {}, n_iter_max=stop + 1, beta=beta)
    for a, b in zip(fa, fb):
        np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-7)
    _, cc, _ = _run(T, F0, {}, n_iter_max=3, beta=beta)
    np.testing.assert_allclose(cc, full[:3], rtol=1e-6)


@pytest.mark.parametrize("beta", [1, 0.5])
def test_ntf_mu_forms_no_tensor_sized_model(beta, monkeypatch):
    """After a warm-up iteration the peak of allocated memory over 3 iterations rises by less than |T| * 4 / 8 bytes; the
    CUDA-core path (NNFAC_NTF_TC=0) allocates more than |T| * 4 bytes for it."""
    import torch
    import nn_fac.ntf as ntf
    T, F0 = _ntf_problem(SHAPE, RANK, 0.4, seed=13)
    tbytes = T.size * 4
    rises = []
    for tc in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTF_TC", tc)
        state = ntf.DeviceNTF(T, F0, torch.float32)
        args = (RANK, 1.0, "mu", beta, [None] * 3, [], [False] * 3)
        state.step_async(*args)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()
        for _ in range(3):
            state.step_async(*args)
        torch.cuda.synchronize()
        rises.append(torch.cuda.max_memory_allocated() - before)
        del state
    assert rises[0] < tbytes / 8, rises
    assert rises[1] > tbytes, rises


# ---------------------------------------------------------------------------------------------
# 3. Routes that keep the CUDA-core update
# ---------------------------------------------------------------------------------------------
def test_four_way_rank65_and_fp32x3_keep_the_old_path(monkeypatch):
    """A 4-way tensor, rank 65 and precision "fp32x3" still match the oracle and form the model tensor (the old path)."""
    import nn_fac.config as config
    import nn_fac.ntf as ntf
    from oracle import nnfac_oracle as orc
    cases = [("4-way", (8, 10, 64, 24), 6, "auto"), ("rank 65", (96, 40, 128), 65, "auto"), ("fp32x3", (24, 24, 24), 4, "fp32x3")]
    for name, shape, r, precision in cases:
        T, F0 = _ntf_problem(shape, r, 0.4, seed=14)
        calls = _count_model(monkeypatch)
        config.set_precision(precision)
        try:
            _, costs, _ = ntf.ntf(T, r, init="custom", factors_0=[f.copy() for f in F0], n_iter_max=4, tol=-1, return_costs=True,
                                  update_rule="mu", beta=1, sparsity_coefficients=[None] * len(shape), fixed_modes=[],
                                  normalize=[False] * len(shape))
        finally:
            config.set_precision("auto")
        ref = orc.compute_ntf(T.astype(np.float64), r, [f.astype(np.float64) for f in F0], n_iter_max=4, tol=-1, update_rule="mu",
                              beta=1)[1]
        assert calls, name
        np.testing.assert_allclose(costs, ref, rtol=1e-4 if precision == "auto" else 1e-6, err_msg=name)
