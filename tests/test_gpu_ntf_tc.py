"""The tensor-core NTF path (DeviceNTF over one copy of the tensor as bf16 hi/lo planes) against float64.

Covers the three kernels only NTF uses: the Khatri-Rao operand written straight into the K-major planes of cross(0, None)
(set_krao), the same product as the rank-contiguous row planes of the fused residual pass (set_krao_rows), and the view plans
that read the unfoldings of the other modes in place (last mode: MN-major operand; middle modes: 3-D TMA map).  Then whole fp32
NTF runs, direct residual or not, against the float64 oracle.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RANKS = [1, 5, 8, 13, 16, 17, 33, 64, 65, 96, 100, 128]


@pytest.fixture(autouse=True)
def _tensor_core_path(fp32_path):
    """Everything in this file is about the float32 kernels, whatever the size of the problem."""
    yield


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _strided(Ft, extra=3):
    """A rank-major factor (r x I) on the device with leading dimension I + extra; the padding columns hold NaN, so that a
    read outside the factor poisons the result."""
    import torch
    r, I = Ft.shape
    buf = torch.full((r, I + extra), float("nan"), dtype=torch.float32, device="cuda")
    buf[:, :I] = _dev(Ft)
    return buf[:, :I]


def _krao_t(At, Bt):
    """Khatri-Rao product of two rank-major fp32 factors, transposed (r x I*J), column a * J + b: one fp32 multiply per
    element, as in the kernels."""
    return (At[:, :, None] * Bt[:, None, :]).reshape(At.shape[0], -1)


def _kind(plan):
    return "view" if getattr(plan, "_base", None) is not None else "full"


def _state(T, r, monkeypatch, views=True):
    """DeviceNTF of a float32 tensor: its plans are the ones an NTF run uses (NNFAC_NTF_VIEWS=0: a copy for every mode >= 1)."""
    import torch
    import nn_fac.ntf as ntf
    monkeypatch.setenv("NNFAC_NTF_VIEWS", "1" if views else "0")
    F = [np.zeros((s, r), np.float32) for s in T.shape]
    state = ntf.DeviceNTF(_dev(T), F, torch.float32)
    monkeypatch.delenv("NNFAC_NTF_VIEWS")
    assert state.plans is not None
    return state


# ---------------------------------------------------------------------------------------------
# 1. Operand installs, bit for bit
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r", RANKS)
def test_set_krao_writes_the_planes_cross_would_split(r):
    """set_krao(At, Bt) + cross(0, None) == cross(0, krao^T) bit for bit, on a full one-sided plan, on a plan whose columns
    are padded (I * J % 64 != 0), and on the middle- and last-mode views of a tensor; on the full plans also
    == set_factor(1, krao^T) + cross(0, None).  I != J everywhere (a swapped slow / fast index shows), strided factors with
    NaN padding (a read outside the factor shows)."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(100 + r)
    shape = (40, 24, 64)
    T = rng.randn(*shape).astype(np.float32)
    Ft = [rng.randn(r, s).astype(np.float32) for s in shape]
    base = ops.NMFPlan(_dev(T).reshape(shape[0], -1)).bind_rank(r, sides=1)
    padded = ops.NMFPlan(_dev(rng.randn(50, 7 * 9).astype(np.float32))).bind_rank(r, sides=1)
    Gt = [rng.randn(r, 7).astype(np.float32), rng.randn(r, 9).astype(np.float32)]
    cases = [("full", base, Ft[1], Ft[2]),
             ("padded", padded, Gt[0], Gt[1]),
             ("middle view", base.view(40, 24, 64, r), Ft[0], Ft[2]),
             ("last view", base.view(40 * 24, 64, 1, r), Ft[0], Ft[1])]
    assert [_kind(c[1]) for c in cases] == ["full", "full", "view", "view"]
    for name, plan, At, Bt in cases:
        Kt = _krao_t(At, Bt)
        plan.set_krao(_strided(At), _strided(Bt))
        got = plan.cross(0, None).clone()
        assert torch.isfinite(got).all(), name
        assert torch.equal(got, plan.cross(0, _dev(Kt))), name
        if _kind(plan) == "full":
            plan.set_factor(1, _dev(Kt))
            assert torch.equal(got, plan.cross(0, None)), name


@pytest.mark.parametrize("r", RANKS)
def test_set_krao_rows_writes_the_row_planes_set_factor_would(r):
    """fused(0, 0) after set_krao_rows(At, Bt) gives the same MTTKRP and the same cost bits as after set_factor(1, krao^T)
    (both write the row planes of factor 1).  A stale operand is installed first: ranks the install skips would keep it."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(200 + r)
    I0, I, J = 150, 24, 40
    T = rng.randn(I0, I * J).astype(np.float32)
    Ft0, At, Bt = (rng.randn(r, s).astype(np.float32) for s in (I0, I, J))
    plan = ops.NMFPlan(_dev(T)).bind_rank(r, sides=1)
    plan.set_factor(0, _dev(Ft0))
    plan.set_factor(1, _dev(rng.randn(r, I * J).astype(np.float32)))
    plan.set_krao_rows(_strided(At), _strided(Bt))
    out1, cost1 = (t.clone() for t in plan.fused(0, 0))
    plan.set_factor(1, _dev(_krao_t(At, Bt)))
    out2, cost2 = plan.fused(0, 0)
    assert torch.isfinite(out1).all() and torch.isfinite(cost1).all()
    assert torch.equal(out1, out2)
    assert torch.equal(cost1, cost2)


# ---------------------------------------------------------------------------------------------
# 2. MTTKRP of every mode against float64, on the plan DeviceNTF picks
# ---------------------------------------------------------------------------------------------
def _mttkrp_bound(T64, mode, Kt64):
    """float64 (unfold(T, mode) @ krao)^T and 3e-5 (|krao|^T |unfold(T, mode)|^T): the 2^-17 representation error of each
    operand in two bf16 planes, the dropped lo * lo term and the fp32 accumulation, on signed data."""
    from oracle import nnfac_oracle as orc
    unf = orc.unfold(T64, mode)
    return Kt64 @ unf.T, 3e-5 * (np.abs(Kt64) @ np.abs(unf).T)


def _krao_operands(Ft, mode):
    """(At, Bt) such that set_krao(At, Bt) installs the Khatri-Rao product of every factor but `mode`'s (first kept factor
    slowest): for a 4-way tensor At is the fp32 Khatri-Rao product of the first two kept factors."""
    kept = [f for i, f in enumerate(Ft) if i != mode]
    At = kept[0]
    for f in kept[1:-1]:
        At = _krao_t(At, f)
    return At, kept[-1]


# per shape, the plan of each mode: "full" (mode 0, or a one-sided plan on a copy of the unfolding) or "view" (in place)
MTTKRP_SHAPES = {
    (64, 96, 72): "full full view",           # last mode I = 72: the second 64-row box of a tile is partial
    (16, 40, 200): "full full view",          # last mode I = 200
    (40, 64, 8): "full full view",            # last mode I = 8
    (24, 5, 128): "full view view",           # middle mode I = 5
    (20, 130, 64): "full view view",          # middle mode I = 130: two row tiles, the second partial; I_0 = 20 < 128
    (130, 8, 64): "full view view",           # I_0 = 130: two row tiles of mode 0
    (6, 10, 64, 128): "full view view view",  # 4-way: two middle views and a last-mode view
    (6, 10, 64, 72): "full view full view",   # 4-way: mode 2 is a copy (right = 72), last mode I = 72
}


@pytest.mark.parametrize("r", [5, 64, 100])
@pytest.mark.parametrize("shape", list(MTTKRP_SHAPES), ids=lambda s: "x".join(map(str, s)))
def test_mttkrp_of_every_mode_matches_float64(shape, r, monkeypatch):
    """set_krao + cross(0, None) on the plan of each mode (as DeviceNTF builds it) against float64, element-wise, signed data.
    Each view also against the copy plan of the same unfolding (NNFAC_NTF_VIEWS=0): same rows, columns and partition, same
    products -> the same bits."""
    import torch
    rng = np.random.RandomState(sum(shape) * 7 + r)
    T = rng.randn(*shape).astype(np.float32)
    Ft = [rng.randn(r, s).astype(np.float32) for s in shape]
    views, copies = _state(T, r, monkeypatch), _state(T, r, monkeypatch, views=False)
    assert " ".join(_kind(p) for p in views.plans) == MTTKRP_SHAPES[shape]
    assert all(_kind(p) == "full" for p in copies.plans)
    T64 = T.astype(np.float64)
    for mode in range(len(shape)):
        At, Bt = _krao_operands(Ft, mode)
        got = []
        for plan in (views.plans[mode], copies.plans[mode]):
            plan.set_krao(_strided(At), _strided(Bt))
            got.append(plan.cross(0, None))
        ref, bound = _mttkrp_bound(T64, mode, _krao_t(At.astype(np.float64), Bt.astype(np.float64)))
        err = np.abs(got[0].cpu().numpy() - ref)
        assert (err <= bound).all(), (mode, float((err / bound).max()))
        assert torch.equal(got[0], got[1]), mode


# ---------------------------------------------------------------------------------------------
# 3. The direct residual ||unfold(T) - F krao^T||^2 of the fused pass
# ---------------------------------------------------------------------------------------------
def _residual_case(T, F, At, Bt):
    """set_factor(0, F^T) + set_krao_rows + fused(0, 0) on a one-sided plan over T (I_0 x I*J); returns the MTTKRP, the cost,
    the float64 cost and its bound."""
    from nn_fac import _ops as ops
    plan = ops.NMFPlan(_dev(T)).bind_rank(F.shape[1], sides=1)
    plan.set_factor(0, _dev(np.ascontiguousarray(F.T)))
    plan.set_krao_rows(_strided(At), _strided(Bt))
    out, cost = plan.fused(0, 0)
    T64, F64 = T.astype(np.float64), F.astype(np.float64)
    Kt64 = _krao_t(At.astype(np.float64), Bt.astype(np.float64))
    M = F64 @ Kt64
    ref = float(((T64 - M) ** 2).sum())
    # per element the model and the data carry an error of at most ~2^-16 S, S = |T| + |F| |krao|^T (two bf16 planes per
    # operand, the dropped lo * lo term, fp32 accumulation): |cost - ref| <= sum 2 |T - M| e + e^2.  2^-14 on the linear term
    # and 2^-30 on the quadratic one (which only matters when the fit is near exact) leave a factor of about 2 to spare.
    S = np.abs(T64) + np.abs(F64) @ np.abs(Kt64)
    bound = 2.0 ** -14 * float((np.abs(T64 - M) * S).sum()) + 2.0 ** -30 * float((S * S).sum())
    return out, float(cost.item()), ref, bound


# Worst |cost - ref| / bound observed over this grid on a B200 (1000 W): 3.5e-3 (rank 5), 6.8e-3 (64), 1.2e-2 (96), 1.4e-2 (128).
# The bound sums absolute values; the errors of the elements largely cancel.
@pytest.mark.parametrize("r", [5, 64, 96, 128])
def test_direct_residual_matches_float64(r):
    """fused(0, 0) on a one-sided plan at rank 5, 64, 96 and 128 (rk = 128: MODE_RES<128> on a one-sided plan): the MTTKRP
    within the bound of section 2, the cost within the residual bound; an exact fit and zero slices / rank columns."""
    rng = np.random.RandomState(300 + r)
    I0, I, J = 150, 24, 40
    F = rng.rand(I0, r).astype(np.float32)
    At, Bt = rng.rand(r, I).astype(np.float32), rng.rand(r, J).astype(np.float32)
    M = (F.astype(np.float64) @ _krao_t(At, Bt).astype(np.float64))
    ratios = []
    for name, T in (("noisy", (M * (1 + 0.1 * rng.randn(*M.shape))).astype(np.float32)),
                    ("signed", rng.randn(*M.shape).astype(np.float32)),
                    ("exact fit", M.astype(np.float32))):
        out, cost, ref, bound = _residual_case(T, F, At, Bt)
        mref, mbound = _mttkrp_bound(T.astype(np.float64).reshape(I0, I, J), 0,
                                     _krao_t(At.astype(np.float64), Bt.astype(np.float64)))
        assert (np.abs(out.cpu().numpy() - mref) <= mbound).all(), name
        assert cost >= 0 and abs(cost - ref) <= bound, (name, cost, ref, bound)
        ratios.append(abs(cost - ref) / bound)
    # a zero slice of the tensor and a zero rank column of F
    T = (M * (1 + 0.1 * rng.randn(*M.shape))).astype(np.float32)
    T[7] = 0
    Fz = F.copy()
    Fz[:, r // 2] = 0
    out, cost, ref, bound = _residual_case(T, Fz, At, Bt)
    assert np.all(out.cpu().numpy()[:, 7] == 0)
    assert cost >= 0 and abs(cost - ref) <= bound, ("zeros", cost, ref, bound)
    ratios.append(abs(cost - ref) / bound)
    print(f"rank {r}: worst |cost - ref| / bound = {max(ratios):.3g}")


# ---------------------------------------------------------------------------------------------
# 4. Whole fp32 NTF runs against the float64 oracle
# ---------------------------------------------------------------------------------------------
NTF_CASES = {
    # name: (shape, rank, keyword arguments, plan of each mode)
    "views": ((96, 40, 128), 16, {}, "full view view"),
    "mixed": ((72, 64, 72), 16, {}, "full full view"),
    "rank96": ((96, 40, 128), 96, {}, "full view view"),
    "sparsity": ((96, 40, 128), 16, dict(sparsity_coefficients=[0.05, None, 0.02]), "full view view"),
    "fixed1": ((72, 64, 72), 16, dict(fixed_modes=[1]), "full full view"),
    "fixed0": ((96, 40, 128), 16, dict(fixed_modes=[0]), "full view view"),   # mode 1, the first free mode, is a view
}


def _ntf_problem(shape, r, sigma, seed):
    """Rank-r CP tensor plus sigma * mean * U[0, 1) noise (float32) and a start near the truth: after 10 HALS iterations the
    normalised objective is ~1e-2 for sigma = 0.4 and ~1e-3 for sigma = 0.12."""
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(seed)
    fs = [rng.rand(s, r) for s in shape]
    low = orc.fold(fs[0] @ orc.khatri_rao(fs, skip_matrix=0).T, 0, shape)
    T = (low + sigma * low.mean() * rng.rand(*shape)).astype(np.float32)
    F0 = [(f * (1 + 0.3 * rng.rand(*f.shape))).astype(np.float32) for f in fs]
    return T, F0


def _run(T, F0, r, kw, n_iter_max=10, tol=-1):
    import nn_fac.ntf as ntf
    nm = T.ndim
    args = dict(sparsity_coefficients=[None] * nm, fixed_modes=[], normalize=[False] * nm)
    args.update({k: list(v) for k, v in kw.items()})
    return ntf.ntf(T, r, init="custom", factors_0=[f.copy() for f in F0], n_iter_max=n_iter_max, tol=tol, return_costs=True,
                   **args)


def _oracle(T, F0, r, kw, n_iter_max=10):
    from oracle import nnfac_oracle as orc
    args = {k: list(v) for k, v in kw.items()}
    return orc.compute_ntf(T.astype(np.float64), r, [f.astype(np.float64) for f in F0], n_iter_max=n_iter_max, tol=-1, **args)[1]


@pytest.mark.parametrize("sigma", [0.4, 0.12], ids=["fit1e-2", "fit1e-3"])
@pytest.mark.parametrize("case", sorted(NTF_CASES))
def test_ntf_fp32_runs_match_float64(case, sigma, monkeypatch):
    """10 iterations of fp32 NTF HALS through the plans DeviceNTF builds (views where the extents allow) against the float64
    oracle from the same fp32 inputs: objective within 1e-4.  The run with a copy for every mode (NNFAC_NTF_VIEWS=0) gives the
    same factors bit for bit and the same costs."""
    import nn_fac.ntf as ntf
    shape, r, kw, kinds = NTF_CASES[case]
    T, F0 = _ntf_problem(shape, r, sigma, seed=len(case) + int(100 * sigma))
    state = _state(T, r, monkeypatch)
    assert " ".join(_kind(p) for p in state.plans) == kinds
    assert state.direct_cost("hals", kw.get("fixed_modes", ()))              # the objective is the direct residual
    del state
    ref = _oracle(T, F0, r, kw)
    fit = 1e-2 if sigma == 0.4 else 1e-3
    assert 0.3 * fit < ref[-1] < 3 * fit
    fa, costs, _ = _run(T, F0, r, kw)
    np.testing.assert_allclose(costs, ref, rtol=1e-4)
    monkeypatch.setenv("NNFAC_NTF_VIEWS", "0")
    fb, copies, _ = _run(T, F0, r, kw)
    for a, b in zip(fa, fb):
        np.testing.assert_array_equal(a, b)
    if kw.get("fixed_modes") == [0]:
        # with views the residual takes an extra pass over unfold(T, 0); with copies it comes from the pass over the copy of
        # unfold(T, 1) that also yields that mode's MTTKRP: the same quantity summed in another order
        np.testing.assert_allclose(copies, costs, rtol=2e-5)
    else:
        np.testing.assert_array_equal(copies, costs)


def test_ntf_fp32_four_way_formula_path_matches_float64():
    """A 4-way tensor (mode 1 a middle view, mode 2 a copy, mode 3 a last-mode view with I = 72): the MTTKRP of every mode on the
    tensor core, the cost by the reference's formula (no direct residual for 4-way tensors).  That formula keeps an absolute
    error of ~8e-7 on the normalised objective (DeviceNTF.direct_cost; 8.4e-7 measured here on a B200): at an objective of
    8e-3 it misses 1e-4 relative (1.03e-4 measured), so this case runs at a fit of 2e-2."""
    import torch
    import nn_fac.ntf as ntf
    shape, r = (6, 10, 64, 72), 8
    T, F0 = _ntf_problem(shape, r, 0.7, seed=4)
    state = ntf.DeviceNTF(T, F0, torch.float32)
    assert " ".join(_kind(p) for p in state.plans) == "full view full view" and not state.direct_cost("hals")
    ref = _oracle(T, F0, r, {})
    assert 1.5e-2 < ref[-1] < 3e-2
    _, costs, _ = _run(T, F0, r, {})
    np.testing.assert_allclose(costs, ref, rtol=1e-4)


def test_ntf_fp32_fixed_mode_0_early_stop_rolls_back_two_iterations():
    """fixed_modes=[0] with the first free mode a view: the direct residual comes from an extra pass over unfold(T, 0).  On a
    stop both speculative iterations are dropped, with and without CUDA-graph replay (as in
    test_gpu_parity.py::test_ntf_fp32_early_stop_rolls_back_two_iterations)."""
    shape, r, kw = (96, 40, 128), 16, dict(fixed_modes=[0])
    T, F0 = _ntf_problem(shape, r, 0.12, seed=5)
    _, full, _ = _run(T, F0, r, kw, n_iter_max=12)
    np.testing.assert_allclose(full, _oracle(T, F0, r, kw, n_iter_max=12), rtol=1e-4)
    tol = 0.5 * (abs(full[5] - full[6]) + abs(full[6] - full[7]))
    stop = next(k for k in range(1, 12) if abs(full[k - 1] - full[k]) < tol)
    assert stop < 11
    fa, ca, _ = _run(T, F0, r, kw, n_iter_max=12, tol=tol)
    assert len(ca) == stop + 1
    np.testing.assert_allclose(ca, full[:stop + 1], rtol=1e-6)
    fb, _, _ = _run(T, F0, r, kw, n_iter_max=stop + 1)                     # the same iterations without a stop
    for a, b in zip(fa, fb):
        np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-7)
    _, cc, _ = _run(T, F0, r, kw, n_iter_max=3)                            # short runs launch eagerly (no graph)
    np.testing.assert_allclose(cc, full[:3], rtol=1e-6)


# ---------------------------------------------------------------------------------------------
# 5. Refusals
# ---------------------------------------------------------------------------------------------
def test_krao_installs_and_views_refuse_what_they_cannot_address():
    import torch
    from nn_fac import _lib as L
    from nn_fac import _ops as ops
    r = 5
    base = ops.NMFPlan(torch.rand((40, 24 * 64), device="cuda")).bind_rank(r, sides=1)
    At, Bt = torch.rand((r, 40), device="cuda"), torch.rand((r, 64), device="cuda")
    view = base.view(40, 24, 64, r)
    assert view is not None
    with pytest.raises(L.NnfacError):
        view.set_krao_rows(At, Bt)                                          # a view has no row planes
    with pytest.raises(L.NnfacError):
        view.set_krao(At, Bt[:, :63])                                       # I * J != n
    with pytest.raises(L.NnfacError):
        base.set_krao(torch.rand((r, 24), device="cuda"), Bt[:, :60])
    mid = ops.NMFPlan(torch.rand((40, 24 * 72), device="cuda")).bind_rank(r, sides=1)
    assert mid.view(40, 24, 72, r) is None                                  # middle mode, right = 72 % 64 != 0
    last = ops.NMFPlan(torch.rand((40, 64 * 12), device="cuda")).bind_rank(r, sides=1)
    assert last.view(40 * 64, 12, 1, r) is None                             # last mode, I = 12 % 8 != 0
