"""NTD on the tensor core over one copy of the tensor (fp32, every rank <= 64) against float64.

DeviceNTD keeps the tensor once, as the bf16 hi/lo planes of the one-sided plan of unfold(T, 0); the other modes read them through
views (or a one-sided plan on a copy where an unfolding cannot be addressed in place), and core_plan reads them as unfold(T, 0)^T
for every contraction over mode 0.  Operands B_n = G x_{j != n} F_j are installed straight from B_n (NMFPlan.set_operand).
Checked here: the install bit for bit, one pass of every plan kind element-wise against float64, whole MU / HALS runs against the
float64 oracle, graph replay, the memory the route takes, and the routes that keep the CUDA-core update.
"""
import numpy as np
import pytest

from tests.test_gpu_ntf_mu_tc import _bounds
from tests.test_gpu_ntf_tc import _dev

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _tensor_core_path(fp32_path):
    """Everything in this file is about the float32 kernels, whatever the size of the problem."""
    yield


def _unfold(a, mode):
    return np.reshape(np.moveaxis(a, mode, 0), (a.shape[mode], -1))


def _split(shape, mode):
    return int(np.prod(shape[:mode])), shape[mode], int(np.prod(shape[mode + 1:]))


def _plans(T, r):
    """DeviceNTD of a float32 tensor with rank r on every mode: (plans of modes 0.., core plan, kind of each)."""
    import torch
    import nn_fac.ntd as ntd
    shape = T.shape
    st = ntd.DeviceNTD(T, np.ones([r] * T.ndim, np.float32), [np.ones((s, r), np.float32) for s in shape], torch.float32)
    kinds = ["base"] + ["view" if getattr(p, "_base", None) is not None else "copy" for p in st.plans[1:]]
    kinds.append("view" if getattr(st.core_plan, "_base", None) is not None else "copy")
    return st, kinds


def _copy_plan(X, r):
    from nn_fac import _ops as ops
    return ops.NMFPlan(_dev(np.ascontiguousarray(X))).bind_rank(r, sides=1)


def _operands(T, mode, r, rng):
    """(X, B, left, right) of the plan of `mode` (None: the core plan): X the unfolding that plan holds (rows x contraction), B the
    operand as a C-order (left, r, right) array, V = B_(mode) its r x contraction unfolding."""
    if mode is None:
        return _unfold(T, 0).T, (rng.rand(1, r, T.shape[0]) + 0.1).astype(np.float32), 1, T.shape[0]
    left, _, right = _split(T.shape, mode)
    return _unfold(T, mode), (rng.rand(left, r, right) + 0.1).astype(np.float32), left, right


def _V(B):
    return B.transpose(1, 0, 2).reshape(B.shape[1], -1)


# ---------------------------------------------------------------------------------------------
# 1. The install, bit for bit
# ---------------------------------------------------------------------------------------------
def test_install_equals_cross_of_the_explicit_unfolding():
    """On the base plan, a middle view, a last view, a copy plan and the core plan, cross(0, None) after set_operand(B) gives the
    bits of cross(0, unfolding of B).  A 3-plane plan and mismatched extents are refused without writing."""
    import torch
    from nn_fac import _lib as L
    from nn_fac import _ops as ops
    rng = np.random.RandomState(1)
    r = 12
    T = (rng.rand(64, 128, 192) + 0.1).astype(np.float32)
    st, kinds = _plans(T, r)
    assert kinds == ["base", "view", "view", "view"]
    cases = [(st.plans[m], m) for m in range(3)] + [(st.core_plan, None), (_copy_plan(_unfold(T, 1), r), 1)]
    for plan, mode in cases:
        _, B, left, right = _operands(T, mode, r, rng)
        Bd = _dev(B)
        plan.set_operand(Bd, left, right)
        got = plan.cross(0, None)
        want = plan.cross(0, _dev(_V(B)))
        assert torch.equal(got, want), mode
        # refused without writing: wrong rank, wrong extents
        with pytest.raises(L.NnfacError):
            plan.set_operand(_dev(np.zeros((left, r + 1, right), np.float32)), left, right)
        with pytest.raises(L.NnfacError):
            plan.set_operand(Bd, left * right, 2)
        assert torch.equal(plan.cross(0, None), want), mode
    three = ops.NMFPlan(_dev(_unfold(T, 0))).bind_rank(r, sides=1, planes=3)
    _, B, left, right = _operands(T, 0, r, rng)
    want = three.cross(0, _dev(_V(B)))
    with pytest.raises(L.NnfacError):
        three.set_operand(_dev(B * 2), left, right)
    assert torch.equal(three.cross(0, None), want)


# ---------------------------------------------------------------------------------------------
# 2. One pass against float64
# ---------------------------------------------------------------------------------------------
# (64, 128, 192): every unfolding a view; (40, 64, 128): views, the core plan contracts over I_0 = 40 < 64 rows;
# (64, 128, 96): mode 1 a copy (trailing extent 96 is not a multiple of 64), mode 2 and the core views;
# (40, 36, 50): padded base planes, every other plan a copy
PASS_SHAPES = {(64, 128, 192): ["base", "view", "view", "view"], (40, 64, 128): ["base", "view", "view", "view"],
               (64, 128, 96): ["base", "copy", "view", "view"], (40, 36, 50): ["base", "copy", "copy", "copy"]}


def _pass(plan, Ft, B, left, right, beta):
    """set_factor_rows(F^T) + set_operand(B) + the pass of the update: (numerator, denominator or None, cost or None) on the host."""
    plan.set_factor_rows(_dev(Ft))
    plan.set_operand(_dev(B), left, right)
    if beta == 2:
        return plan.cross(0, None).cpu().numpy(), None, None
    if beta == 1:
        num, cost = plan.fused(0, 1, want_cost=True)
        return num.cpu().numpy(), None, float(cost.item())
    cost = plan.fused_beta(0, beta, want_cost=True)
    return plan.reduce(0).cpu().numpy(), plan.reduce_den(0).cpu().numpy(), float(cost.item())


@pytest.mark.parametrize("beta", [1, 2, 0, 0.5, 3])
@pytest.mark.parametrize("r", [5, 33, 64])
@pytest.mark.parametrize("shape", list(PASS_SHAPES), ids=lambda s: "x".join(map(str, s)))
def test_pass_of_every_plan_matches_float64(shape, r, beta):
    """The pass of every plan (base, views or copies of modes 1 and 2, the core plan) against float64 element by element, with the
    bounds of the NTF passes; the denominator summed by reduce_den.  A view gives the bits of the copy plan of the same unfolding,
    and a second run the bits of the first."""
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(sum(shape) + 10 * r + int(10 * beta))
    T = (rng.rand(*shape) + 0.1).astype(np.float32)
    st, kinds = _plans(T, r)
    assert kinds == PASS_SHAPES[shape]
    for idx, (plan, mode) in enumerate([(st.plans[m], m) for m in range(3)] + [(st.core_plan, None)]):
        X, B, left, right = _operands(T, mode, r, rng)
        Ft = (rng.rand(r, X.shape[0]) + 0.1).astype(np.float32)
        got = _pass(plan, Ft, B, left, right, beta)
        again = _pass(plan, Ft, B, left, right, beta)
        X64, V64, F64 = X.astype(np.float64), _V(B).astype(np.float64), Ft.T.astype(np.float64)
        K = F64 @ V64
        num64 = (((K ** (beta - 2.0)) * X64) @ V64.T).T
        den64 = ((K ** (beta - 1.0)) @ V64.T).T
        nb, db, cb = _bounds(num64, den64, X64, K, 0, beta)
        err = np.abs(got[0] - num64)
        assert (err <= nb).all(), (kinds[idx], mode, "numerator", float((err / nb).max()))
        if got[1] is not None:
            err = np.abs(got[1] - den64)
            assert (err <= db).all(), (kinds[idx], mode, "denominator", float((err / db).max()))
        if got[2] is not None:
            assert abs(got[2] - orc.beta_divergence(X64, K, beta)) <= cb, (kinds[idx], mode, got[2])
            assert got[2] == again[2]
        for a, b in zip(got[:2], again[:2]):
            if a is not None:
                np.testing.assert_array_equal(a, b)
        if kinds[idx] == "view":
            copy = _pass(_copy_plan(X, r), Ft, B, left, right, beta)
            for a, b in zip(got[:2], copy[:2]):
                if a is not None:
                    np.testing.assert_array_equal(a, b)
            if beta not in (1, 2):
                assert got[2] == copy[2]
            elif beta == 1:     # the cost adds the sum of X, which each plan forms over its own layout
                assert abs(got[2] - copy[2]) <= 1e-6 * float(X64.sum())
    if beta == 2:
        # the cost of beta = 2: half the direct residual of one fused pass on the base plan
        base = st.plans[0]
        X, B, left, right = _operands(T, 0, r, rng)
        Ft = (rng.rand(r, X.shape[0]) + 0.1).astype(np.float32)
        base.set_factor(0, _dev(Ft))
        base.set_factor(1, _dev(_V(B)))
        _, res = base.fused(0, 0)
        K = Ft.T.astype(np.float64) @ _V(B).astype(np.float64)
        ref = float(((X.astype(np.float64) - K) ** 2).sum())
        assert abs(float(res.item()) - ref) <= 1e-4 * ref


# ---------------------------------------------------------------------------------------------
# 3. Whole runs against the float64 oracle
# ---------------------------------------------------------------------------------------------
def _problem(shape, ranks, seed):
    rng = np.random.RandomState(seed)
    sub = "abcd,ia,jb,kc,ld->ijkl" if len(shape) == 4 else "abc,ia,jb,kc->ijk"
    Fs = [rng.rand(s, r) for s, r in zip(shape, ranks)]
    T = np.einsum(sub, rng.rand(*ranks), *Fs)
    T = (T + 0.1 * T.mean() * rng.rand(*shape) + 1e-3).astype(np.float32)
    G0 = rng.rand(*ranks).astype(np.float32)
    F0 = [rng.rand(s, r).astype(np.float32) for s, r in zip(shape, ranks)]
    return T, G0, F0


RUN_CASES = {
    "views": ((64, 128, 192), [8, 12, 10], {}),
    "copies": ((40, 36, 50), [6, 5, 7], {}),
    "fixed0": ((64, 128, 192), [8, 12, 10], dict(fixed_modes=[0])),
    "fixed_last": ((64, 128, 192), [8, 12, 10], dict(fixed_modes=[2])),
    "normalized_core": ((64, 128, 192), [8, 12, 10], dict(normalize=[False] * 3 + [True], mode_core_norm=1)),
    "4way": ((14, 12, 16, 10), [3, 4, 2, 3], {}),
}


def _run_ntd(T, G0, F0, kw, rule, beta=2, n_iter_max=8, tol=0):
    import nn_fac.ntd as ntd
    nm = T.ndim
    args = dict(sparsity_coefficients=[None] * (nm + 1), fixed_modes=[], normalize=[False] * (nm + 1), mode_core_norm=None)
    args.update({k: (list(v) if isinstance(v, list) else v) for k, v in kw.items()})
    return ntd.ntd(T, [int(s) for s in G0.shape], init="custom", core_0=G0.copy(), factors_0=[f.copy() for f in F0],
                   n_iter_max=n_iter_max, tol=tol, update_rule=rule, beta=beta, return_costs=True, deterministic=True, **args)


def _spy_plans(monkeypatch):
    """Records whether each DeviceNTD built the tensor-core plans."""
    import nn_fac.ntd as ntd
    built = []
    orig = ntd.DeviceNTD.__init__

    def init(self, *a, **k):
        orig(self, *a, **k)
        built.append(self.plans is not None)
    monkeypatch.setattr(ntd.DeviceNTD, "__init__", init)
    return built


@pytest.mark.parametrize("beta", [0, 0.5, 1, 1.5, 2, 3])
@pytest.mark.parametrize("case", list(RUN_CASES))
def test_ntd_mu_runs_match_float64(case, beta, monkeypatch):
    """8 iterations of ntd(update_rule="mu") from fp32 inputs on the tensor core against the float64 oracle: the objective within
    1e-4 relative at every iteration; fixed factors stay as they were."""
    from oracle import nnfac_oracle as orc
    shape, ranks, kw = RUN_CASES[case]
    T, G0, F0 = _problem(shape, ranks, seed=5)
    built = _spy_plans(monkeypatch)
    _, factors, costs, _ = _run_ntd(T, G0, F0, kw, "mu", beta)
    assert built == [True]
    okw = {k: v for k, v in kw.items()}
    _, _, ref = orc.compute_ntd_mu(T.astype(np.float64), G0.astype(np.float64), [f.astype(np.float64) for f in F0], n_iter_max=8,
                                   tol=0, beta=beta, **okw)
    assert len(costs) == 8
    np.testing.assert_allclose(costs, ref, rtol=1e-4)
    for m in kw.get("fixed_modes", []):
        np.testing.assert_array_equal(factors[m], F0[m])


@pytest.mark.parametrize("case", ["views", "4way", "fixed0"])
def test_ntd_hals_runs_match_float64(case, monkeypatch):
    """ntd(update_rule="hals") with every contraction over mode 0 on the core plan, against the float64 oracle within 1e-4."""
    from oracle import nnfac_oracle as orc
    shape, ranks, kw = RUN_CASES[case]
    T, G0, F0 = _problem(shape, ranks, seed=6)
    built = _spy_plans(monkeypatch)
    _, _, costs, _ = _run_ntd(T, G0, F0, kw, "hals", n_iter_max=5)
    assert built == [True]
    _, _, ref = orc.compute_ntd_hals(T.astype(np.float64), G0.astype(np.float64), [f.astype(np.float64) for f in F0], n_iter_max=5,
                                     tol=0, **kw)
    np.testing.assert_allclose(costs, ref, rtol=1e-4)


# ---------------------------------------------------------------------------------------------
# 4. Graph replay
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0, 2])
def test_graph_replay_equals_eager_iterations(beta, monkeypatch):
    """compute_ntd (MU) replays the outer iteration from a CUDA graph: the same costs, core and factors bit for bit as eager
    launches, for a fixed iteration count and when the stop test drops the speculative iteration."""
    T, G0, F0 = _problem((64, 128, 192), [8, 12, 10], seed=7)
    res = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTD_GRAPH", flag)
        core, factors, costs, _ = _run_ntd(T, G0, F0, {}, "mu", beta, n_iter_max=12)
        tol = abs(costs[4] - costs[5]) * 1.01
        core_s, factors_s, costs_s, _ = _run_ntd(T, G0, F0, {}, "mu", beta, n_iter_max=12, tol=tol)
        res[flag] = (core, factors, costs, core_s, factors_s, costs_s)
    a, b = res["1"], res["0"]
    assert 2 <= len(a[5]) <= 6 and a[5] == a[2][:len(a[5])]
    assert a[2] == b[2] and a[5] == b[5]
    for i in (0, 3):
        np.testing.assert_array_equal(a[i], b[i])
    for i in (1, 4):
        for x, y in zip(a[i], b[i]):
            np.testing.assert_array_equal(x, y)


# ---------------------------------------------------------------------------------------------
# 5. Memory
# ---------------------------------------------------------------------------------------------
def _device_problem(size, rank, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    T = torch.rand((size,) * 3, device="cuda", generator=g) + 0.1
    G = torch.rand((rank,) * 3, device="cuda", generator=g)
    F = [torch.rand((size, rank), device="cuda", generator=g) for _ in range(3)]
    return T, G, F


def test_plans_hold_less_than_16_bytes_per_element():
    """At 256^3 / 32^3 the plans' workspaces (planes, operand planes, partials, denominator buffers) together hold less than 16
    bytes per tensor element; a two-sided plan per mode took 24 for the planes alone."""
    import torch
    import nn_fac.ntd as ntd
    T, G, F = _device_problem(256, 32, 1)
    st = ntd.DeviceNTD(T, G, F, torch.float32)
    st.step_mu_async(0, [], [False] * 4, None)                     # allocates the denominator buffers of the general-beta passes
    torch.cuda.synchronize()
    held = 0
    for p in st.plans + [st.core_plan]:
        held += p._workspace.numel()
        held += 0 if p._den is None else p._den.numel() * 4
        held += 0 if p._xf32 is None else p._xf32.numel()
    assert held < 16 * T.numel(), held / T.numel()
    print(f"plans: {held / T.numel():.2f} bytes per element")


@pytest.mark.parametrize("beta", [0, 2])
def test_mu_iterations_form_no_tensor_sized_temporary(beta, monkeypatch):
    """After a warm-up iteration the peak of allocated memory over 3 MU iterations rises by less than |T| * 4 / 8 bytes (256^3,
    core 8^3); the CUDA-core route (NNFAC_NTD_TC=0) allocates more than |T| * 4 bytes for it."""
    import torch
    import nn_fac.ntd as ntd
    T, G, F = _device_problem(256, 8, 2)
    tbytes = T.numel() * 4
    rises = []
    for tc in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTD_TC", tc)
        st = ntd.DeviceNTD(T, G, F, torch.float32)
        assert (st.plans is not None) == (tc == "1")
        st.step_mu_async(beta, [], [False] * 4, None)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()
        for _ in range(3):
            st.step_mu_async(beta, [], [False] * 4, None)
        torch.cuda.synchronize()
        rises.append(torch.cuda.max_memory_allocated() - before)
        del st
    assert rises[0] < tbytes / 8, rises
    assert rises[1] > tbytes, rises


def test_tensor_core_route_never_forms_the_element_wise_terms(monkeypatch):
    """ops.mu_terms (K^(beta-2) * T and K^(beta-1) on tensors of the size of T) is never called on the tensor-core route, for any
    beta; the CUDA-core route calls it."""
    from nn_fac import _ops as ops
    calls = []
    orig = ops.mu_terms
    monkeypatch.setattr(ops, "mu_terms", lambda *a, **k: calls.append(1) or orig(*a, **k))
    T, G0, F0 = _problem((64, 128, 192), [8, 12, 10], seed=8)
    for beta in (0, 0.5, 1, 1.5, 3):
        _run_ntd(T, G0, F0, {}, "mu", beta, n_iter_max=3)
    assert not calls
    monkeypatch.setenv("NNFAC_NTD_TC", "0")
    _run_ntd(T, G0, F0, {}, "mu", 0, n_iter_max=2)
    assert calls


# ---------------------------------------------------------------------------------------------
# 6. Fallbacks
# ---------------------------------------------------------------------------------------------
def test_out_of_memory_for_the_plans_takes_the_cuda_core_route(monkeypatch):
    """No memory for the plans (NMFPlan.bind_rank raising OutOfMemoryError): the CUDA-core route, with the objective of
    NNFAC_NTD_TC=0."""
    import torch
    from nn_fac import _ops as ops
    T, G0, F0 = _problem((64, 128, 192), [8, 12, 10], seed=9)
    monkeypatch.setenv("NNFAC_NTD_TC", "0")
    _, _, want, _ = _run_ntd(T, G0, F0, {}, "mu", 0.5, n_iter_max=4)
    monkeypatch.delenv("NNFAC_NTD_TC")

    def no_memory(self, *a, **k):
        raise torch.cuda.OutOfMemoryError("no memory for the plan")
    monkeypatch.setattr(ops.NMFPlan, "bind_rank", no_memory)
    built = _spy_plans(monkeypatch)
    _, _, got, _ = _run_ntd(T, G0, F0, {}, "mu", 0.5, n_iter_max=4)
    assert built == [False]
    assert got == want


def test_rank65_float64_and_fp32x3_build_no_plans(monkeypatch):
    import nn_fac.config as config
    T, G0, F0 = _problem((70, 24, 32), [65, 4, 4], seed=10)
    built = _spy_plans(monkeypatch)
    _run_ntd(T, G0, F0, {}, "mu", 1, n_iter_max=2)
    T, G0, F0 = _problem((64, 128, 192), [8, 12, 10], seed=10)
    _run_ntd(T.astype(np.float64), G0.astype(np.float64), [f.astype(np.float64) for f in F0], {}, "mu", 1, n_iter_max=2)
    config.set_precision("fp32x3")
    try:
        _run_ntd(T, G0, F0, {}, "mu", 1, n_iter_max=2)
    finally:
        config.set_precision("auto")
    assert built == [False, False, False]
