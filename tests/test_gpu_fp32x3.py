"""GPU tests of precision "fp32x3": 3-plane tensor-core NMF (X and the factors as hi + mid + lo bf16 planes, six-term products)
and the float64 route it takes everywhere else.

Printed lines starting with "fp32x3:" carry the measured errors (run with -s to see them)."""
import numpy as np
import pytest
import torch

from oracle import nnfac_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _auto_precision():
    import nn_fac.config as config
    config.set_precision("auto")
    yield
    config.set_precision("auto")


def _f32(x):
    return np.asarray(x).astype(np.float32)


def _plan(X, r, planes):
    from nn_fac import _ops as ops
    return ops.NMFPlan(torch.as_tensor(X).cuda()).bind_rank(r, planes=planes)


# ---------------------------------------------------------------------------------------------
# exact ingest
# ---------------------------------------------------------------------------------------------
def test_three_planes_hold_the_fp32_values_exactly():
    rng = np.random.RandomState(7)
    m, n = 256, 192
    X = _f32(10.0 ** rng.uniform(-20, 20, size=(m, n)))
    X[rng.rand(m, n) < 0.1] = 0.0
    big = np.finfo(np.float32).max
    X[0, :4] = [big, np.nextafter(big, 0, dtype=np.float32), _f32(3.39e38)[()], _f32(2.0 ** 128 - 2.0 ** 119)[()]]   # hi would overflow bf16
    X[1, :2] = [np.finfo(np.float32).tiny, _f32(1.2345678e-32)[()]]                # small values whose lo stays normal
    plan = _plan(X, 16, 3)
    plan.enable_f32()
    torch.cuda.synchronize()
    buf = plan._xf32
    side0 = buf[:m * n * 4].view(torch.int32).view(m, n).cpu().numpy()
    off1 = (m * n * 4 + 255) // 256 * 256
    side1 = buf[off1:off1 + n * m * 4].view(torch.int32).view(n, m).cpu().numpy()
    bits = X.view(np.int32)
    np.testing.assert_array_equal(side0, bits)
    np.testing.assert_array_equal(side1, bits.T)


# ---------------------------------------------------------------------------------------------
# kernel precision at a near-exact point
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def near_exact():
    rng = np.random.RandomState(11)
    m = n = 4096
    r = 32
    U = _f32(rng.rand(m, r))
    V = _f32(rng.rand(r, n))
    X = _f32((U.astype(np.float64) @ V.astype(np.float64)) * (1.0 + 1e-3 * rng.uniform(-1, 1, size=(m, n))))
    dev = torch.device("cuda")
    U64, V64, X64 = (torch.as_tensor(a, device=dev).double() for a in (U, V, X))
    K = U64 @ V64
    ref = {"res": float(((X64 - K) ** 2).sum()), "kl": float((X64 * torch.log(X64 / K) - X64 + K).sum()),
           "VXt": (V64 @ X64.T), "UtX": (U64.T @ X64)}
    del K
    out = {}
    for planes in (2, 3):
        plan = _plan(X, r, planes)
        plan.set_factor(0, torch.as_tensor(U.T.copy(), device=dev))
        plan.set_factor(1, torch.as_tensor(V, device=dev))
        VXt, c_res = plan.fused(0, 0)
        _, c_kl = plan.fused(0, 1)
        UtX = plan.cross(1, None)
        torch.cuda.synchronize()
        rel = lambda a, b: float(torch.linalg.norm(a.double() - b) / torch.linalg.norm(b))  # noqa: E731
        out[planes] = {"res": abs(float(c_res) - ref["res"]) / ref["res"], "kl": abs(float(c_kl) - ref["kl"]) / ref["kl"],
                       "VXt": rel(VXt, ref["VXt"]), "UtX": rel(UtX, ref["UtX"])}
        del plan
    for k in ("res", "kl", "VXt", "UtX"):
        print(f"fp32x3: near-exact 4096^2 r=32 {k}: 2 planes rel.err {out[2][k]:.3e}, 3 planes {out[3][k]:.3e}")
    return out


@pytest.mark.parametrize("term", ["res", "kl"])
def test_cost_terms_with_three_planes(near_exact, term):
    """The residual isolates the third plane.  For KL most of the gap comes from the 3-plane pass summing the terms k g(x/k)
    directly: the 2-plane cost formula cancels at this point (DESIGN.md section 1), so this checks the 3-plane pass as a whole."""
    e2, e3 = near_exact[2][term], near_exact[3][term]
    assert e3 <= 1e-6, (term, e3)
    assert 8 * e3 <= e2, (term, e2, e3)


@pytest.mark.parametrize("term", ["VXt", "UtX"])
def test_cross_products_with_three_planes(near_exact, term):
    assert near_exact[3][term] <= near_exact[2][term], (term, near_exact[2][term], near_exact[3][term])


# ---------------------------------------------------------------------------------------------
# acceptance: 4096 x 4096, rank 32, near-exact data, 100 iterations
# ---------------------------------------------------------------------------------------------
RULES = {"hals": ("hals", 2), "mu1": ("mu", 1), "mu2": ("mu", 2)}


@pytest.fixture(scope="module")
def c1_like():
    rng = np.random.RandomState(2024)
    m = n = 4096
    r = 32
    data = _f32(rng.rand(m, r) @ rng.rand(r, n) + 1e-2 * rng.rand(m, n))
    U0, V0 = _f32(rng.rand(m, r)), _f32(rng.rand(r, n))
    refs = {}
    for tag, (rule, beta) in RULES.items():
        refs[tag] = np.asarray(orc.compute_nmf(data.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64), n_iter_max=100,
                                               tol=0, update_rule=rule, beta=beta)[2])
    return data, U0, V0, r, refs


def _run(c1_like, tag, precision, monkeypatch):
    import nn_fac.config as config
    import nn_fac.nmf as nmf
    from nn_fac import _fast
    data, U0, V0, r, refs = c1_like
    rule, beta = RULES[tag]
    seen = []
    init = _fast.CudaEngine.__init__

    def spy(self, X, rank, device=None, planes=2):
        init(self, X, rank, device, planes=planes)
        seen.append(self.plan.planes)
    monkeypatch.setattr(_fast.CudaEngine, "__init__", spy)
    config.set_precision(precision)
    try:
        U, V, costs, _ = nmf.nmf(data, r, init="custom", U_0=U0, V_0=V0, n_iter_max=100, tol=0, update_rule=rule, beta=beta,
                                 return_costs=True)
    finally:
        config.set_precision("auto")
    ref = refs[tag]
    dev = np.abs(np.asarray(costs) - ref) / ref
    return U, V, dev, seen


@pytest.mark.parametrize("tc_sweep", [False, True])
def test_acceptance_hals(c1_like, tc_sweep, monkeypatch):
    """The HALS solves of fp32x3 run on the fp32 CUDA-core sweep (the default, asserted); the tensor-core sweep, whose step
    operand is a bf16 hi/lo split, is run too and its deviation reported."""
    from nn_fac import _fast
    default = _fast.TC_SWEEP_FP32X3
    monkeypatch.setattr(_fast, "TC_SWEEP_FP32X3", tc_sweep)
    U, V, dev, planes = _run(c1_like, "hals", "fp32x3", monkeypatch)
    print(f"fp32x3: acceptance hals ({'tensor-core' if tc_sweep else 'CUDA-core'} sweep): worst rel. deviation over iterations "
          f">= 10: {dev[10:].max():.3e} (at iteration {10 + int(dev[10:].argmax())}), last {dev[-1]:.3e}")
    assert planes == [3]
    assert U.dtype == np.float32 and V.dtype == np.float32
    if tc_sweep == default:
        assert dev[10:].max() <= 1e-4


@pytest.mark.parametrize("tag", ["mu1", "mu2"])
def test_acceptance_mu(c1_like, tag, monkeypatch):
    U, V, dev, planes = _run(c1_like, tag, "fp32x3", monkeypatch)
    print(f"fp32x3: acceptance {tag}: worst rel. deviation over iterations >= 10: {dev[10:].max():.3e} "
          f"(at iteration {10 + int(dev[10:].argmax())}), last {dev[-1]:.3e}")
    assert planes == [3]
    assert U.dtype == np.float32 and V.dtype == np.float32
    assert dev[10:].max() <= 1e-4


@pytest.mark.parametrize("tag", sorted(RULES))
def test_fp32_deviation_is_reported(c1_like, tag, monkeypatch):
    """The same problem on the 2-plane path: the deviation is printed, not asserted."""
    _, _, dev, planes = _run(c1_like, tag, "fp32", monkeypatch)
    print(f"fp32x3: same problem under 'fp32' ({tag}): worst rel. deviation over iterations >= 10: {dev[10:].max():.3e}, "
          f"last {dev[-1]:.3e}")
    assert planes == [2]


# ---------------------------------------------------------------------------------------------
# the float64 route, the sharded refusal, and no state carried between modes
# ---------------------------------------------------------------------------------------------
def _fp32x3():
    import nn_fac.config as config
    config.set_precision("fp32x3")


def test_nmf_rank_96_takes_the_float64_route():
    import nn_fac.nmf as nmf
    rng = np.random.RandomState(96)
    m, n, r = 300, 200, 96
    data = _f32(rng.rand(m, 8) @ rng.rand(8, n) + 0.1 * rng.rand(m, n))
    U0, V0 = _f32(rng.rand(m, r)), _f32(rng.rand(r, n))
    _fp32x3()
    for rule, beta in (("hals", 2), ("mu", 1)):
        U, V, costs, _ = nmf.nmf(data, r, init="custom", U_0=U0, V_0=V0, n_iter_max=4, tol=0, update_rule=rule, beta=beta,
                                 return_costs=True)
        ref = orc.compute_nmf(data.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64), n_iter_max=4, tol=0,
                              update_rule=rule, beta=beta)[2]
        assert U.dtype == np.float32 and V.dtype == np.float32
        np.testing.assert_allclose(costs, ref, rtol=1e-6)


def test_one_nmf_step_takes_the_float64_route():
    import nn_fac.nmf as nmf
    rng = np.random.RandomState(5)
    m, n, r = 120, 90, 6
    data = _f32(rng.rand(m, n))
    U0, V0 = _f32(rng.rand(m, r)), _f32(rng.rand(r, n))
    _fp32x3()
    U, V, cost = nmf.one_nmf_step(data, r, U0, V0, np.linalg.norm(data), "hals", 2, [None, None], [], [False, False], True)
    Ur, Vr, cref = orc.one_nmf_step(data.astype(np.float64), U0.astype(np.float64), V0.astype(np.float64))
    assert U.dtype == np.float32 and V.dtype == np.float32
    np.testing.assert_allclose(cost, cref, rtol=1e-6)
    np.testing.assert_allclose(U, Ur, rtol=1e-6, atol=1e-7)


def test_ntf_and_ntd_take_the_float64_route():
    import nn_fac.ntd as ntd
    import nn_fac.ntf as ntf
    rng = np.random.RandomState(3)
    I, r = 24, 4
    T = _f32(np.einsum("ir,jr,kr->ijk", rng.rand(I, r), rng.rand(I, r), rng.rand(I, r)) + 0.05 * rng.rand(I, I, I))
    F0 = [_f32(rng.rand(I, r)) for _ in range(3)]
    _fp32x3()
    factors, costs, _ = ntf.ntf(T, r, init="custom", factors_0=F0, n_iter_max=3, tol=-1, return_costs=True,
                                sparsity_coefficients=[None] * 3, normalize=[False] * 3)
    ref = orc.compute_ntf(T.astype(np.float64), r, [f.astype(np.float64) for f in F0], n_iter_max=3, tol=0)[1]
    assert all(np.asarray(f).dtype == np.float32 for f in factors)
    np.testing.assert_allclose(costs, ref, rtol=1e-6)
    G0 = _f32(rng.rand(r, r, r))
    out = ntd.ntd(T, [r] * 3, init="custom", core_0=G0, factors_0=F0, n_iter_max=2, tol=0, update_rule="mu", beta=1,
                  sparsity_coefficients=[None] * 4, fixed_modes=[], normalize=[False] * 4, return_costs=True, deterministic=True)
    ref = orc.compute_ntd_mu(T.astype(np.float64), G0.astype(np.float64), [f.astype(np.float64) for f in F0], n_iter_max=2, tol=0,
                             beta=1)[2]
    assert np.asarray(out[0]).dtype == np.float32
    np.testing.assert_allclose(out[2], ref, rtol=1e-6)


def test_sharded_refuses_fp32x3():
    from nn_fac import sharded
    rng = np.random.RandomState(1)
    _fp32x3()
    with pytest.raises(NotImplementedError):
        sharded.compute_nmf_sharded(_f32(rng.rand(256, 256)), 8, _f32(rng.rand(256, 8)), _f32(rng.rand(8, 256)), n_iter_max=2)


def test_no_state_leaks_between_modes():
    import nn_fac.config as config
    import nn_fac.nmf as nmf
    rng = np.random.RandomState(9)
    m, n, r = 640, 512, 16
    data = _f32(rng.rand(m, r) @ rng.rand(r, n) + 0.05 * rng.rand(m, n))
    U0, V0 = _f32(rng.rand(m, r)), _f32(rng.rand(r, n))

    def run(precision, rule, beta):
        config.set_precision(precision)
        try:
            return nmf.nmf(data, r, init="custom", U_0=U0, V_0=V0, n_iter_max=6, tol=0, update_rule=rule, beta=beta,
                           return_costs=True)[2]
        finally:
            config.set_precision("auto")
    for rule, beta in (("hals", 2), ("mu", 1)):
        before = run("fp32", rule, beta)
        run("fp32x3", rule, beta)
        after = run("fp32", rule, beta)
        np.testing.assert_array_equal(before, after)


def test_update_rules_and_one_step_functions_return_float32():
    """Direct calls of the update rules, the one-step NTF / NTD functions and PARAFAC2 compute in float64 under fp32x3 and hand
    back float32: the float64 results ("fp64") rounded to float32."""
    import nn_fac.config as config
    import nn_fac.ntd as ntd
    import nn_fac.ntf as ntf
    import nn_fac.parafac2 as p2
    import nn_fac.update_rules.mu as mu
    import nn_fac.update_rules.nnls as nnls
    rng = np.random.RandomState(21)
    r, n, I = 5, 40, 12
    A = rng.rand(30, r)
    UtU, UtM, V0, Vt = A.T @ A, A.T @ rng.rand(30, n), rng.rand(r, n), rng.rand(r, n)
    X, U, V = rng.rand(30, n), rng.rand(30, r), rng.rand(r, n)
    T = np.einsum("ir,jr,kr->ijk", rng.rand(I, 3), rng.rand(I, 3), rng.rand(I, 3)) + 0.05 * rng.rand(I, I, I)
    F = [rng.rand(I, 3) for _ in range(3)]
    G = rng.rand(3, 3, 3)
    slices = [rng.rand(10, 8) for _ in range(3)]
    calls = {
        "hals_nnls_acc": lambda: [nnls.hals_nnls_acc(UtM, UtU, V0, maxiter=50)[0]],
        "hals_coupling_nnls_acc": lambda: [nnls.hals_coupling_nnls_acc(UtM, UtU, V0, Vt, 0.3, maxiter=50)[0]],
        "switch_alternate_mu": lambda: [mu.switch_alternate_mu(X, U, V, 1, "U"), mu.switch_alternate_mu(X, U, V, 2, "V")],
        "mu_betadivmin": lambda: [mu.mu_betadivmin(U, V, X, 1.5)],
        "mu_tensorial": lambda: [mu.mu_tensorial(G, F, T, 1)],
        "one_ntf_step": lambda: ntf.one_ntf_step([T.reshape(I, -1)], 3, F, np.linalg.norm(T), "hals", 2, [None] * 3, [],
                                                 [False] * 3)[0],
        "one_ntd_step": lambda: (lambda o: [o[0]] + list(o[1]))(ntd.one_ntd_step(T, [3] * 3, G, F, np.linalg.norm(T), [None] * 4, [],
                                                                                 [False] * 4, None)),
        "one_ntd_step_mu": lambda: (lambda o: [o[0]] + list(o[1]))(ntd.one_ntd_step_mu(T, [3] * 3, G, F, 1, np.linalg.norm(T), [],
                                                                                       [False] * 4, None)),
        "parafac_2": lambda: (lambda o: list(o[0]) + [o[1]] + list(o[2]))(p2.parafac_2(slices, 2, True, init="random", n_iter_max=2,
                                                                                        tol=0, deterministic=True, seed=3)),
    }
    for name, call in calls.items():
        config.set_precision("fp64")
        ref = [np.asarray(a) for a in call()]
        _fp32x3()
        got = call()
        config.set_precision("auto")
        for a, b in zip(got, ref):
            assert isinstance(a, np.ndarray) and a.dtype == np.float32, (name, type(a), getattr(a, "dtype", None))
            assert b.dtype == np.float64, name
            np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-30, err_msg=name)
