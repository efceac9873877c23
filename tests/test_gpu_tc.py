"""tcgen05 / TMA cross-product kernel (fp32 headline path) against a float64 host product."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _tensor_core_path(fp32_path):
    """Everything in this file is about the float32 kernels, whatever the size of the problem."""
    yield


@pytest.mark.parametrize("m,n,r", [(128, 64, 16), (256, 512, 64), (1000, 500, 10), (777, 1300, 33), (4096, 2048, 128),
                                   (130, 70, 9)])
def test_plan_cross_matches_float64(m, n, r):
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(m + n + r)
    X = rng.rand(m, n).astype(np.float32)
    V = rng.rand(r, n).astype(np.float32)
    Ut = rng.rand(r, m).astype(np.float32)
    plan = ops.NMFPlan(torch.from_numpy(X).cuda()).bind_rank(r)
    vmt = plan.cross(0, torch.from_numpy(V).cuda()).cpu().numpy()
    utm = plan.cross(1, torch.from_numpy(Ut).cuda()).cpu().numpy()
    ref0 = V.astype(np.float64) @ X.astype(np.float64).T
    ref1 = Ut.astype(np.float64) @ X.astype(np.float64)
    # bf16x2 split operands (2^-17 relative per element, unbiased) + fp32 accumulation
    np.testing.assert_allclose(vmt, ref0, rtol=2e-5)
    np.testing.assert_allclose(utm, ref1, rtol=2e-5)
    # typical error is far below the bound
    assert np.abs(vmt / ref0 - 1).mean() < 2e-6
    assert np.abs(utm / ref1 - 1).mean() < 2e-6


def test_plan_cross_is_deterministic_and_linear():
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(0)
    X = torch.from_numpy(rng.rand(1500, 900).astype(np.float32)).cuda()
    V = torch.from_numpy(rng.rand(24, 900).astype(np.float32)).cuda()
    plan = ops.NMFPlan(X).bind_rank(24)
    a = plan.cross(0, V).clone()
    b = plan.cross(0, V).clone()
    assert torch.equal(a, b)
    c = plan.cross(0, 2.0 * V)
    torch.testing.assert_close(c, 2.0 * a, rtol=1e-6, atol=0)


@pytest.mark.parametrize("m,n,r", [(128, 64, 16), (384, 320, 64), (1000, 500, 10), (777, 1300, 33), (2048, 4096, 64)])
def test_fused_pass_matches_float64(m, n, r):
    """Fused X pass (model tile formed and consumed on chip) against float64 numpy, both sides, both modes."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(m * 7 + n + r)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    X = ((rng.rand(m, r) @ rng.rand(r, n)) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)
    plan = ops.NMFPlan(torch.from_numpy(X).cuda()).bind_rank(r)
    plan.set_factor(0, torch.from_numpy(np.ascontiguousarray(U.T)).cuda())
    plan.set_factor(1, torch.from_numpy(V).cuda())
    X64, U64, V64 = X.astype(np.float64), U.astype(np.float64), V.astype(np.float64)
    K = U64 @ V64
    # mode 0: cross products + squared residual
    out, cost = plan.fused(0, 0)
    np.testing.assert_allclose(out.cpu().numpy(), V64 @ X64.T, rtol=2e-5)
    np.testing.assert_allclose(cost.item(), np.sum((X64 - K) ** 2), rtol=2e-5)
    out, cost = plan.fused(1, 0)
    np.testing.assert_allclose(out.cpu().numpy(), U64.T @ X64, rtol=2e-5)
    np.testing.assert_allclose(cost.item(), np.sum((X64 - K) ** 2), rtol=2e-5)
    # mode 1: beta = 1 numerators + KL divergence
    kl = np.sum(X64 * np.log(X64 / K) - X64 + K)
    out, cost = plan.fused(0, 1)
    np.testing.assert_allclose(out.cpu().numpy(), V64 @ (X64 / K).T, rtol=3e-5)
    np.testing.assert_allclose(cost.item(), kl, rtol=2e-5)
    out, cost = plan.fused(1, 1)
    np.testing.assert_allclose(out.cpu().numpy(), U64.T @ (X64 / K), rtol=3e-5)
    np.testing.assert_allclose(cost.item(), kl, rtol=2e-5)


@pytest.mark.parametrize("m,n,r", [(384, 320, 96), (1000, 520, 128), (777, 1300, 80), (2048, 4096, 128), (130, 70, 65)])
def test_fused_pass_rank_65_to_128_matches_float64(m, n, r):
    """Residual + cross-product pass at padded rank 128 (two 64-rank atoms per factor slab, 128-wide contraction, rows of the
    aligned factor loaded global -> tensor memory) against float64 numpy, both sides; ragged tiles and ranks."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(m * 7 + n + r)
    U = rng.rand(m, r).astype(np.float32) + 0.05
    V = rng.rand(r, n).astype(np.float32) + 0.05
    X = ((rng.rand(m, r) @ rng.rand(r, n)) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)
    plan = ops.NMFPlan(torch.from_numpy(X).cuda()).bind_rank(r)
    plan.set_factor(0, torch.from_numpy(np.ascontiguousarray(U.T)).cuda())
    plan.set_factor(1, torch.from_numpy(V).cuda())
    X64, U64, V64 = X.astype(np.float64), U.astype(np.float64), V.astype(np.float64)
    K = U64 @ V64
    for side, ref in ((0, V64 @ X64.T), (1, U64.T @ X64)):
        out, cost = plan.fused(side, 0)
        np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=2e-5)
        np.testing.assert_allclose(cost.item(), np.sum((X64 - K) ** 2), rtol=2e-5)
        # the split partials left in the plan add up to the same numbers
        plan.fused(side, 0, keep_partials=True)
        np.testing.assert_array_equal(plan.reduce(side).cpu().numpy(), out.cpu().numpy())
    with pytest.raises(Exception):
        plan.fused(0, 1)                              # the beta = 1 pass covers rank <= 64


@pytest.mark.parametrize("r,length,dtype", [(10, 500, "float64"), (64, 65536, "float32"), (33, 1301, "float32"),
                                            (64, 8192, "float64"), (1, 7, "float32"), (96, 700, "float32"),
                                            (128, 70000, "float32"), (65, 33, "float32"), (100, 5000, "float64")])
def test_gram_matches_float64(r, length, dtype):
    """F F^T of a rank-major factor (nmf.py:407 / :432); 64 < r <= 128 in fp32: 64 x 64 block pairs, else the general kernel."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(r + length)
    F = rng.rand(r, length).astype(dtype)
    ref = F.astype(np.float64) @ F.astype(np.float64).T
    Fd = torch.from_numpy(F).cuda()
    out = ops.gram(Fd)
    np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-12 if dtype == "float64" else 3e-6)
    assert torch.equal(out, ops.gram(Fd))                                    # deterministic
    # strided view (the column slice a rank owns in the sharded U solve)
    if length > 300:
        sub = Fd[:, 128:300]
        np.testing.assert_allclose(ops.gram(sub).cpu().numpy(), F[:, 128:300].astype(np.float64) @ F[:, 128:300].astype(np.float64).T,
                                   rtol=1e-12 if dtype == "float64" else 3e-6)


@pytest.mark.parametrize("x_source", ["planes", "f32"])
@pytest.mark.parametrize("m,n,r", [(384, 320, 64), (1000, 500, 10), (777, 1300, 33)])
def test_mu_finish_equals_reduce_apply_install(m, n, r, x_source, monkeypatch):
    """The one-kernel finish of a beta=1 update (split partials -> ratio -> clamp -> planes) against the separate
    reduce / mu_apply / set_factor kernels, both factors; then the next fused pass must see the new factor.  x_source: the beta = 1
    pass rebuilds X from the bf16 planes (NNFAC_MU_F32=0, what runs when X is too large for the copies) or reads the fp32 copies."""
    import torch
    from nn_fac import _ops as ops
    monkeypatch.setenv("NNFAC_MU_F32", "0" if x_source == "planes" else "1")
    rng = np.random.RandomState(m + n + r)
    U = (rng.rand(m, r) + 0.05).astype(np.float32)
    V = (rng.rand(r, n) + 0.05).astype(np.float32)
    X = ((rng.rand(m, r) @ rng.rand(r, n)) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)
    Ut_d, V_d = torch.from_numpy(np.ascontiguousarray(U.T)).cuda(), torch.from_numpy(V).cuda()
    plans = [ops.NMFPlan(torch.from_numpy(X).cuda()).bind_rank(r) for _ in range(2)]
    for p in plans:
        p.set_factor(0, Ut_d)
        p.set_factor(1, V_d)
    for which, F, other in ((0, Ut_d, V_d), (1, V_d, Ut_d)):
        den = ops.row_sums(other)
        num, _ = plans[0].fused(which, 1, want_cost=False)
        ref = ops.mu_apply(F, num, den_vec=den, vec_per_row=True, gamma=1.0, floor=1e-12)
        plans[0].set_factor(which, ref)
        plans[1].fused(which, 1, want_cost=False, keep_partials=True)
        new = plans[1].mu_finish(which, F, den, 1e-12)
        assert torch.equal(new, ref)
        a, ca = plans[0].fused(1 - which, 1)
        b, cb = plans[1].fused(1 - which, 1)
        assert torch.equal(a, b) and torch.equal(ca, cb)
    assert all((p._xf32 is None) == (x_source == "planes") for p in plans)


# ---------------------------------------------------------------------------------------------
# tensor-core HALS sweep (tc_sweep_kernel): shapes, edge cases and full parity of the stop rule
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r,n,maxiter", [(64, 130, 100), (64, 20000, 100), (40, 777, 100), (17, 4096, 100), (1, 300, 50),
                                         (64, 1, 30), (33, 5000, 1), (64, 3000, 2), (48, 70000, 7),
                                         (128, 5000, 100), (96, 777, 100), (100, 30000, 100), (128, 130, 100), (65, 300, 3),
                                         (128, 37000, 20), (80, 1, 30)])
def test_tc_sweep_matches_oracle(r, n, maxiter):
    """fp32 tcgen05 solve vs the float64 oracle on identical inputs: same sweep count (one flip near the threshold is
    allowed), solution to fp32 accuracy, ragged tiles / partial warps / partial rank blocks."""
    import nn_fac.update_rules.nnls as nnls
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(7 * r + n)
    m = 2 * r + 3
    U = rng.rand(m, r)
    M = U @ rng.rand(r, n) + 0.1 * rng.rand(m, n)
    UtM, UtU, V0 = (U.T @ M).astype(np.float32), (U.T @ U).astype(np.float32), rng.rand(r, n).astype(np.float32)
    V, eps, cnt, _ = nnls.hals_nnls_acc(UtM, UtU, V0, maxiter=maxiter, delta=0.01)
    Vo, eps_o, cnt_o, _ = orc.hals_nnls_acc(UtM.astype(np.float64), UtU.astype(np.float64), V0.astype(np.float64),
                                            maxiter=maxiter, delta=0.01)
    assert V.dtype == np.float32 and V.shape == V0.shape
    assert abs(cnt - cnt_o) <= 1
    if cnt == cnt_o:
        assert np.linalg.norm(V - Vo) <= 5e-4 * np.linalg.norm(Vo)
        if eps_o > 1e-8 * np.sum(Vo ** 2):           # a fully converged solve ends on rounding noise (e.g. r = 1)
            assert abs(eps - eps_o) <= 2e-3 * abs(eps_o)
    assert (V >= 0).all()


def test_tc_sweep_zero_diagonal_row_is_left_alone():
    """nnls.py:160: a row whose diagonal entry of UtU is zero is skipped -- even when its initial value is negative."""
    import nn_fac.update_rules.nnls as nnls
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(3)
    r, n = 20, 500
    U = rng.rand(50, r)
    U[:, 5] = 0.0                                     # column 5 of U is zero -> row/column 5 of UtU is zero
    UtU = (U.T @ U).astype(np.float32)
    UtM = (U.T @ (U @ rng.rand(r, n) + 0.05 * rng.rand(50, n))).astype(np.float32)
    V0 = rng.rand(r, n).astype(np.float32)
    V0[5, ::2] *= -1.0
    V, _, cnt, _ = nnls.hals_nnls_acc(UtM, UtU, V0, maxiter=40, delta=0.01)
    Vo, _, cnt_o, _ = orc.hals_nnls_acc(UtM.astype(np.float64), UtU.astype(np.float64), V0.astype(np.float64), maxiter=40,
                                        delta=0.01)
    np.testing.assert_array_equal(V[5], V0[5])
    assert abs(cnt - cnt_o) <= 1
    if cnt == cnt_o:
        assert np.linalg.norm(V - Vo) <= 5e-4 * np.linalg.norm(Vo)


def test_tc_sweep_is_deterministic_and_pure():
    import torch
    from nn_fac import _ops as ops
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    r, n = 64, 40000
    U = torch.rand((150, r), generator=g, device="cuda")
    G = (U.T @ U).contiguous()
    b = (G @ torch.rand((r, n), generator=g, device="cuda")).contiguous()
    V0 = torch.rand((r, n), generator=g, device="cuda")
    outs = []
    for _ in range(3):
        V = V0.clone()
        st = ops.hals_nnls(b, G, V, r, 100, 0.01, 0.0, False, False).clone()
        outs.append((V, st))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][0], outs[2][0])
    assert torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("r,n,maxiter,delta", [(64, 8192, 100, 0.01), (64, 8192, 60, 0.0), (40, 9000, 100, 0.01), (64, 30000, 100, 0.01),
                                               (128, 12000, 100, 0.01), (96, 20000, 37, 0.0), (64, 8192, 1, 0.01), (64, 8192, 2, 0.01),
                                               (64, 300, 100, 0.01), (17, 8192, 3, 0.5)])
def test_tc_sweep_lagged_stop_test_is_bit_identical(r, n, maxiter, delta):
    """The stop test of nnls.py:156 evaluated with a lag of one sweep (the whole next sweep runs speculatively and is undone
    when the test ends the solve, nnfac_ctx_sweep_variant) executes the same sweeps as the plain variant: same bits, same
    count, same eps -- including maxiter = 1, 2 (nothing to speculate on) and early stops."""
    import torch
    from nn_fac import _lib as L
    from nn_fac import _ops as ops
    g = torch.Generator(device="cuda"); g.manual_seed(11 * r + n)
    U = torch.rand((2 * r + 5, r), generator=g, device="cuda")
    G = (U.T @ U).contiguous()
    b = (G @ torch.rand((r, n), generator=g, device="cuda") + 0.1 * torch.rand((r, n), generator=g, device="cuda")).contiguous()
    V0 = torch.rand((r, n), generator=g, device="cuda")
    lib, ctx = L.load_library(), L.ctx(V0.device)
    outs = []
    try:
        for mode in (0, 2):
            L.check(lib.nnfac_ctx_sweep_variant(ctx, mode))
            V = V0.clone()
            st = ops.hals_nnls(b, G, V, r, maxiter, delta, 0.0, False, False).clone()
            outs.append((V, st))
    finally:
        L.check(lib.nnfac_ctx_sweep_variant(ctx, -1))
    assert torch.equal(outs[0][1], outs[1][1]), (outs[0][1], outs[1][1])
    assert torch.equal(outs[0][0], outs[1][0])
    assert 2 <= int(outs[0][1][1].item()) <= maxiter + 1


# ---------------------------------------------------------------------------------------------
# plan plumbing: caller workspace, slab-wise ingest of a host array, reuse of installed planes, fp32 copies
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_plan_from_host_equals_plan_from_device(dtype):
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(11)
    m, n, r = 3001, 1700, 24
    X = rng.rand(m, n).astype(dtype)
    V = torch.from_numpy(rng.rand(r, n).astype(np.float32)).cuda()
    dev_plan = ops.NMFPlan(torch.from_numpy(X.astype(np.float32)).cuda()).bind_rank(r)
    old = ops.NMFPlan.SLAB_BYTES
    ops.NMFPlan.SLAB_BYTES = 1 << 20                # many slabs, ragged last one
    try:
        host_plan = ops.NMFPlan(X).bind_rank(r)
    finally:
        ops.NMFPlan.SLAB_BYTES = old
    for which, F in ((0, V), (1, torch.from_numpy(rng.rand(r, m).astype(np.float32)).cuda())):
        assert torch.equal(dev_plan.cross(which, F), host_plan.cross(which, F))


def test_cross_reuses_installed_planes_and_f32_copies_change_nothing(monkeypatch):
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(12)
    m, n, r = 1024, 2304, 48
    X = torch.from_numpy((rng.rand(m, r) @ rng.rand(r, n) + 0.3 * rng.rand(m, n)).astype(np.float32)).cuda()
    Ut = torch.from_numpy(rng.rand(r, m).astype(np.float32)).cuda()
    V = torch.from_numpy(rng.rand(r, n).astype(np.float32)).cuda()
    plan = ops.NMFPlan(X).bind_rank(r)
    plan.set_factor(0, Ut)
    plan.set_factor(1, V)
    assert torch.equal(plan.cross(1, None), plan.cross(1, Ut))
    assert torch.equal(plan.cross(0, None), plan.cross(0, V))
    # the reference reads X from the bf16 planes: without NNFAC_MU_F32=0 the first beta = 1 pass would make the fp32 copies itself
    # and the comparison below would be the copy path against itself
    monkeypatch.setenv("NNFAC_MU_F32", "0")
    ref = [(o.clone(), c.clone()) for o, c in (plan.fused(0, 1), plan.fused(1, 1))]
    assert plan._xf32 is None
    plan.enable_f32()
    for side in (0, 1):
        out, cost = plan.fused(side, 1)
        assert torch.equal(out, ref[side][0]) and torch.equal(cost, ref[side][1])


def test_ntf_tensor_core_mttkrp_matches_generic_path(monkeypatch):
    import torch
    import nn_fac.ntf as ntf
    rng = np.random.RandomState(13)
    shape, r = (60, 45, 70), 12
    fs = [rng.rand(s, r) for s in shape]
    T = (np.einsum("ir,jr,kr->ijk", *fs) + 0.05 * rng.rand(*shape)).astype(np.float32)
    F0 = [rng.rand(s, r).astype(np.float32) for s in shape]
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTF_TC", flag)
        _, costs, _ = ntf.ntf(T, r, init="custom", factors_0=[f.copy() for f in F0], n_iter_max=6, tol=0, return_costs=True)
        out[flag] = costs
    # the reference's cost formula (ntf.py:470) subtracts numbers of the size of ||T||^2: in fp32 both paths carry an
    # absolute noise of ~1e-6 ||T||^2 on a normalised cost of ~1e-3
    np.testing.assert_allclose(out["1"], out["0"], rtol=5e-3)
    assert out["1"][-1] < out["1"][0]


@pytest.mark.parametrize("beta", [1, 2])
def test_ntd_mu_fp32_objective(beta, monkeypatch):
    """fp32 NTD (beta = 1: factor updates through the fused tcgen05 pass) against the float64 oracle, and against the
    generic fp32 path: objective within 1e-4 relative after 8 iterations."""
    import nn_fac.ntd as ntd
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(21)
    shape, ranks = (40, 36, 50), [6, 5, 7]
    G = rng.rand(*ranks)
    Fs = [rng.rand(s, r) for s, r in zip(shape, ranks)]
    T = np.einsum("abc,ia,jb,kc->ijk", G, *Fs) + 0.05 * rng.rand(*shape) + 1e-3
    G0, F0 = rng.rand(*ranks), [rng.rand(s, r) for s, r in zip(shape, ranks)]
    _, _, ref = orc.compute_ntd_mu(T, G0, F0, n_iter_max=8, tol=0, beta=beta)
    f32 = lambda x: x.astype(np.float32)  # noqa: E731
    res = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTD_TC", flag)
        _, _, costs, _ = ntd.ntd(f32(T), list(ranks), init="custom", core_0=f32(G0), factors_0=[f32(f) for f in F0], n_iter_max=8,
                                 tol=0, update_rule="mu", beta=beta, sparsity_coefficients=[None] * 4, fixed_modes=[],
                                 normalize=[False] * 4, return_costs=True, deterministic=True)
        res[flag] = costs
        assert abs(costs[-1] - ref[-1]) <= 1e-4 * abs(ref[-1])
    np.testing.assert_allclose(res["1"], res["0"], rtol=1e-4)


def test_solve_from_split_partials_equals_solve_from_reduced_rhs():
    """nnfac_nmf_plan_hals_solve(UtM = NULL) adds the split-K partials of the last X pass in the reduction kernel's
    order: bit-identical to reducing first; nnfac_nmf_plan_reduce returns that reduced right-hand side."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(31)
    m, n, r = 6000, 4096, 40
    X = torch.from_numpy((rng.rand(m, r) @ rng.rand(r, n) + 0.3 * rng.rand(m, n)).astype(np.float32)).cuda()
    Ut = torch.from_numpy(rng.rand(r, m).astype(np.float32)).cuda()
    V = torch.from_numpy(rng.rand(r, n).astype(np.float32)).cuda()
    plan = ops.NMFPlan(X).bind_rank(r)
    plan.set_factor(0, Ut)
    plan.set_factor(1, V)
    G = ops.gram(V)
    res = torch.zeros(4, dtype=torch.float64, device="cuda")
    rhs, _ = plan.fused(0, 0)                                    # reduced V X^T
    a = plan.hals_solve(0, rhs, G, Ut, 100, 0.01, 0.0, res)
    sweeps_a = res.clone()
    plan.set_factor(0, Ut)                                       # the solve installed its result: put U back
    plan.fused(0, 0, keep_partials=True)                         # partials stay in the plan
    assert torch.equal(plan.reduce(0), rhs)
    b = plan.hals_solve(0, None, G, Ut, 100, 0.01, 0.0, res)
    assert a is not None and b is not None
    assert torch.equal(a, b) and torch.equal(res, sweeps_a)
    # second side through the plain cross product
    plan.set_factor(0, Ut)
    rhs1 = plan.cross(1, None)
    plan.cross(1, None, keep_partials=True)
    assert torch.equal(plan.reduce(1), rhs1)


def test_core_pg_step_state_machine():
    """ntd.py:607-617 on the device: min(step * gradient, core) update, ||delta|| stop test, no-op once done."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(5)
    for dt in (torch.float64, torch.float32):
        core = torch.from_numpy(rng.rand(6, 5, 4)).to(dt).cuda()
        MtX = torch.from_numpy(rng.rand(6, 5, 4)).to(dt).cuda()
        P = torch.from_numpy(rng.rand(6, 5, 4)).to(dt).cuda()
        c = core.double().cpu().numpy().copy()
        g = -MtX.double().cpu().numpy() + P.double().cpu().numpy() + 0.01
        state = torch.tensor([0.0, 1.0, 1.0, 0.0], dtype=torch.float64, device="cuda")
        ops.core_pg_step(core, MtX, P, 0.3, 0.01, 0.01, state)
        d = np.minimum(0.3 * g, c)
        tol = dict(rtol=1e-12) if dt == torch.float64 else dict(rtol=2e-6, atol=1e-7)
        np.testing.assert_allclose(core.double().cpu().numpy(), c - d, **tol)
        st = state.cpu().numpy()
        np.testing.assert_allclose(st[0], np.sqrt((d ** 2).sum()), rtol=1e-6)
        assert st[2] == 2.0 and st[3] == 0.0 and st[0] == st[1]
        # a vanishing second step ends the loop; further calls leave the core alone
        Pz = MtX - 0.01
        ops.core_pg_step(core, MtX, Pz, 0.3, 0.01, 0.01, state)          # gradient = 0 -> upd = 0 < delta * upd_0
        assert state[3].item() == 1.0
        before = core.clone()
        ops.core_pg_step(core, MtX, P, 0.3, 0.01, 0.01, state)
        assert torch.equal(core, before)
        # a first step of size 0 (ntd.py:594 rounds the step to 6 decimals): the reference repeats the no-op 300 times;
        # here they are counted, not executed
        state0 = torch.tensor([0.0, 1.0, 1.0, 0.0], dtype=torch.float64, device="cuda")
        ops.core_pg_step(core, MtX, P, 0.0, 0.0, 0.01, state0)
        assert torch.equal(core, before) and state0.tolist() == [0.0, 0.0, 301.0, 1.0]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_graph_replayed_iterations_equal_eager_iterations(dtype, monkeypatch):
    """compute_ntd (MU) / compute_ntf replay the outer iteration from a CUDA graph from the second iteration on
    (nn_fac/_graph.py): same costs and same results bit for bit as launching every iteration kernel by kernel, both for a
    fixed iteration count and when the reference's stop test (ntd.py:421 / ntf.py:337) drops the speculative iteration."""
    import nn_fac.ntd as ntd
    import nn_fac.ntf as ntf
    rng = np.random.RandomState(3)
    shape, ranks = (40, 36, 50), [6, 5, 7]
    Fs = [rng.rand(s, r) for s, r in zip(shape, ranks)]
    T = (np.einsum("abc,ia,jb,kc->ijk", rng.rand(*ranks), *Fs) + 0.05 * rng.rand(*shape) + 1e-3).astype(dtype)
    G0, F0 = rng.rand(*ranks).astype(dtype), [rng.rand(s, r).astype(dtype) for s, r in zip(shape, ranks)]
    C0 = [rng.rand(s, 8).astype(dtype) for s in shape]

    def run_ntd(tol):
        return ntd.ntd(T, list(ranks), init="custom", core_0=G0.copy(), factors_0=[f.copy() for f in F0], n_iter_max=12, tol=tol,
                       update_rule="mu", beta=1, sparsity_coefficients=[None] * 4, fixed_modes=[], normalize=[False] * 4,
                       return_costs=True, deterministic=True)

    def run_ntf(tol):
        return ntf.ntf(T, 8, init="custom", factors_0=[f.copy() for f in C0], n_iter_max=12, tol=tol, return_costs=True,
                       sparsity_coefficients=[None] * 3, fixed_modes=[], normalize=[False] * 3)

    def run_ntd_hals():
        return ntd.ntd(T, list(ranks), init="custom", core_0=G0.copy(), factors_0=[f.copy() for f in F0], n_iter_max=4, tol=0,
                       update_rule="hals", sparsity_coefficients=[None] * 4, fixed_modes=[], normalize=[False] * 4,
                       return_costs=True, deterministic=True)

    res, hals = {}, {}
    for flag in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTD_GRAPH", flag)
        monkeypatch.setenv("NNFAC_NTF_GRAPH", flag)
        hals[flag] = run_ntd_hals()                          # core loop of ntd.py:607-617 as graph replays from iteration 2
        core, factors, costs, _ = run_ntd(0)
        tol = abs(costs[4] - costs[5]) * 1.01                # the stop test fires at the sixth cost at the latest
        core_s, factors_s, costs_s, _ = run_ntd(tol)
        fac, fcosts, _ = run_ntf(0)
        ftol = abs(fcosts[4] - fcosts[5]) * 1.01
        fac_s, fcosts_s, _ = run_ntf(ftol)
        res[flag] = (core, factors, costs, core_s, factors_s, costs_s, fac, fcosts, fac_s, fcosts_s)
    assert hals["1"][2] == hals["0"][2]
    np.testing.assert_array_equal(hals["1"][0], hals["0"][0])
    for x, y in zip(hals["1"][1], hals["0"][1]):
        np.testing.assert_array_equal(x, y)
    a, b = res["1"], res["0"]
    assert 2 <= len(a[5]) <= 6 and 2 <= len(a[9]) <= 6
    assert a[2] == b[2] and a[5] == b[5] and a[7] == b[7] and a[9] == b[9]
    for i in (0, 3):
        np.testing.assert_array_equal(a[i], b[i])
    for i in (1, 4, 6, 8):
        for x, y in zip(a[i], b[i]):
            np.testing.assert_array_equal(x, y)
    # the early-stopped run returns the state of the iteration whose cost fired the test: a prefix of the full trajectory
    assert a[5] == a[2][:len(a[5])] and a[9] == a[7][:len(a[9])]


@pytest.mark.parametrize("dt_name", ["float32", "float64"])
@pytest.mark.parametrize("ranks", [(32, 32, 32), (9, 9, 3), (64, 17, 40)])
def test_core_pg_step3_equals_mode_products_plus_step(dt_name, ranks):
    """nnfac_core_pg_step3 (two kernels per projected-gradient step of ntd.py:607-617) against the generic route:
    P = core x_n MtM_n by three mode products, then nnfac_core_pg_step."""
    import torch
    from nn_fac import _ops as ops
    dt = getattr(torch, dt_name)
    rng = np.random.RandomState(17)
    core0 = torch.from_numpy(rng.rand(*ranks)).to(dt).cuda()
    MtX = torch.from_numpy(rng.rand(*ranks) * 30).to(dt).cuda()
    MtM = []
    for r in ranks:
        F = rng.rand(50, r)
        MtM.append(torch.from_numpy(F.T @ F).to(dt).cuda().contiguous())
    step = 1.0 / float(np.prod([np.linalg.svd(M.double().cpu().numpy(), compute_uv=False)[0] for M in MtM]))
    a, b = core0.clone(), core0.clone()
    sa = torch.tensor([0.0, 1.0, 1.0, 0.0], dtype=torch.float64, device="cuda")
    sb = torch.tensor([0.0, 1.0, 1.0, 0.0, step, 0.02], dtype=torch.float64, device="cuda")
    Z = torch.empty_like(b)
    for _ in range(5):
        P = ops.multi_mode_dot(a, MtM)
        ops.core_pg_step(a, MtX, P, step, 0.02, 0.01, sa)
        ops.core_pg_step3(b, MtX, MtM, Z, 0.0, 0.0, 0.01, sb, dev_scalars=True)
    tol = dict(rtol=1e-11, atol=1e-13) if dt == torch.float64 else dict(rtol=2e-4, atol=1e-6)
    np.testing.assert_allclose(b.double().cpu().numpy(), a.double().cpu().numpy(), **tol)
    np.testing.assert_allclose(sb[:3].cpu().numpy(), sa[:3].cpu().numpy(), rtol=1e-9 if dt == torch.float64 else 1e-4)
    assert sb[3].item() == sa[3].item() and (a != core0).any()


@pytest.mark.parametrize("case", ["fixed0", "fixed2", "4way", "normalized_core"])
def test_ntd_mu_fp32_variants_vs_oracle(case):
    """fp32 NTD-MU beta = 1 on the tcgen05 path (fused factor passes, fused core-update contraction, shared cost / mode-0
    pass, graph replay) for the cases that change which pass is shared with which: a fixed first or last mode, a 4-way
    tensor (generic core step), a normalised core.  Objective within 1e-4 relative of the float64 oracle after 8 iterations."""
    import nn_fac.ntd as ntd
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(29)
    if case == "4way":
        shape, ranks = (14, 12, 16, 10), [3, 4, 2, 3]
        sub = "abcd,ia,jb,kc,ld->ijkl"
    else:
        shape, ranks = (40, 36, 50), [6, 5, 7]
        sub = "abc,ia,jb,kc->ijk"
    nm = len(shape)
    Fs = [rng.rand(s, r) for s, r in zip(shape, ranks)]
    T = np.einsum(sub, rng.rand(*ranks), *Fs) + 0.05 * rng.rand(*shape) + 1e-3
    G0, F0 = rng.rand(*ranks), [rng.rand(s, r) for s, r in zip(shape, ranks)]
    fixed = {"fixed0": [0], "fixed2": [2]}.get(case, [])
    normalize = [False] * nm + [case == "normalized_core"]
    mcn = 1 if case == "normalized_core" else None
    _, _, ref = orc.compute_ntd_mu(T, G0, F0, n_iter_max=8, tol=0, beta=1, fixed_modes=fixed, normalize=normalize, mode_core_norm=mcn)
    f32 = lambda x: x.astype(np.float32)  # noqa: E731
    core, factors, costs, _ = ntd.ntd(f32(T), list(ranks), init="custom", core_0=f32(G0), factors_0=[f32(f) for f in F0], n_iter_max=8,
                                      tol=0, update_rule="mu", beta=1, sparsity_coefficients=[None] * (nm + 1), fixed_modes=list(fixed),
                                      normalize=list(normalize), mode_core_norm=mcn, return_costs=True, deterministic=True)
    assert len(costs) == 8
    np.testing.assert_allclose(costs, ref, rtol=1e-4)
    for m in fixed:
        np.testing.assert_array_equal(factors[m], f32(F0[m]))


@pytest.mark.parametrize("nway", [3, 4])
def test_ntd_hals_fp32_tensor_core_contraction_matches_generic_path(nway, monkeypatch):
    """ntd(update_rule="hals") in fp32: T x_j F_j^T (ntd.py:550) through the tcgen05 cross product over the planes of an
    unfolding against the strided CUDA-core route (NNFAC_NTD_TC=0), and against the float64 oracle."""
    import nn_fac.ntd as ntd
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(41)
    if nway == 4:
        shape, ranks, sub = (14, 12, 16, 10), [3, 4, 2, 3], "abcd,ia,jb,kc,ld->ijkl"
    else:
        shape, ranks, sub = (40, 36, 50), [6, 5, 7], "abc,ia,jb,kc->ijk"
    Fs = [rng.rand(s, r) for s, r in zip(shape, ranks)]
    T = np.einsum(sub, rng.rand(*ranks), *Fs) + 0.05 * rng.rand(*shape)
    G0, F0 = rng.rand(*ranks), [rng.rand(s, r) for s, r in zip(shape, ranks)]
    _, _, ref = orc.compute_ntd_hals(T, G0, F0, n_iter_max=5, tol=0)
    f32 = lambda x: x.astype(np.float32)  # noqa: E731
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("NNFAC_NTD_TC", flag)
        _, _, costs, _ = ntd.ntd(f32(T), list(ranks), init="custom", core_0=f32(G0), factors_0=[f32(f) for f in F0], n_iter_max=5, tol=0,
                                 update_rule="hals", sparsity_coefficients=[None] * (nway + 1), fixed_modes=[],
                                 normalize=[False] * (nway + 1), return_costs=True, deterministic=True)
        out[flag] = costs
        if flag == "1":
            # with the plans the cost is the direct residual of a fused pass (DeviceNTD.step_hals_async): north-star tolerance
            np.testing.assert_allclose(costs, ref, rtol=1e-4)
        else:
            # CUDA-core route: the reference's own formula (ntd.py:637) in fp32 -- ~1e-6 ||T||^2 of cancellation noise
            np.testing.assert_allclose(costs, ref, atol=3e-6, rtol=2e-2)
    np.testing.assert_allclose(out["1"], out["0"], atol=3e-6, rtol=2e-2)


def test_nmf_hals_more_columns_than_the_tensor_core_solve_covers():
    """m beyond 512 columns per SM: the U solve falls back from the tcgen05 sweep to the CUDA-core sweep, which needs the
    REDUCED right-hand side although the X pass left split-K partials in the plan (nnfac_nmf_plan_reduce)."""
    import nn_fac.nmf as nmf
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(8)
    m, n, r = 80000, 192, 8
    X = rng.rand(m, r) @ rng.rand(r, n) + 0.2 * rng.rand(m, n)
    U0, V0 = rng.rand(m, r), rng.rand(r, n)
    _, _, ref, _ = orc.compute_nmf(X, U0, V0, n_iter_max=4, tol=0, update_rule="hals")
    f32 = lambda x: x.astype(np.float32)  # noqa: E731
    _, _, costs, _ = nmf.nmf(f32(X), r, init="custom", U_0=f32(U0), V_0=f32(V0), n_iter_max=4, tol=0, update_rule="hals",
                             return_costs=True, deterministic=True)
    np.testing.assert_allclose(costs, ref[:len(costs)], rtol=1e-4)


@pytest.mark.parametrize("r", [96, 128])
def test_nmf_hals_rank_65_to_128_fast_path_vs_oracle(r):
    """HALS NMF at rank 65..128 on the tcgen05 path (fused residual pass, cross product, tensor-core sweep with 256 tensor-memory
    columns per tile) against the float64 oracle at a reduced C3 shape: objective @1e-4, sweep counts +-1."""
    import torch
    from nn_fac import _fast
    from oracle import nnfac_oracle as orc
    rng = np.random.RandomState(r)
    m, n = 4096, 2048
    low = rng.rand(m, r) @ rng.rand(r, n)
    X = low + low.mean() * rng.rand(m, n)
    U0, V0 = rng.rand(m, r), rng.rand(r, n)
    stats = {}
    _, _, ref, _ = orc.compute_nmf(X, U0, V0, n_iter_max=4, tol=0, update_rule="hals", stats=stats)
    f32 = lambda x: torch.from_numpy(x.astype(np.float32)).cuda()  # noqa: E731
    assert _fast.eligible(torch.float32, r, "hals", 2)
    st = _fast.FusedNMF(f32(X), f32(U0), f32(V0))
    costs, _ = st.run(4, 0.0, "hals")
    np.testing.assert_allclose(costs, ref, rtol=1e-4)
    got = np.array([t.cpu().numpy() for t in st.sweep_log])          # [iteration][U, V]
    want = np.stack([stats["sweeps_U"], stats["sweeps_V"]], axis=1)
    assert np.abs(got - want).max() <= 1, (got, want)
    # the public entry point takes the same path
    import nn_fac.nmf as nmf
    _, _, c2, _ = nmf.nmf(X.astype(np.float32), r, init="custom", U_0=U0.astype(np.float32), V_0=V0.astype(np.float32),
                          n_iter_max=4, tol=0, update_rule="hals", return_costs=True, deterministic=True)
    np.testing.assert_allclose(c2, costs, rtol=1e-12)


def test_philox_blocks_equal_numpy_restatement_and_tile():
    """Counter-based synthetic data (csrc/synth.cu): device blocks equal the numpy restatement bit for bit, and a matrix
    generated as one block equals the same matrix generated shard by shard."""
    import torch
    from nn_fac import _ops as ops
    from oracle import philox
    full = ops.philox_uniform(300, 517, seed=1234567890123, stream_id=3).cpu().numpy()
    np.testing.assert_array_equal(full, philox.uniform(300, 517, seed=1234567890123, stream_id=3))
    part = ops.philox_uniform(100, 200, row0=150, col0=300, seed=1234567890123, stream_id=3).cpu().numpy()
    np.testing.assert_array_equal(part, full[150:250, 300:500])
    acc = torch.ones((100, 200), device="cuda")
    ops.philox_uniform(100, 200, row0=150, col0=300, seed=1234567890123, stream_id=3, scale=2.0, out=acc, accumulate=True)
    np.testing.assert_allclose(acc.cpu().numpy(), 1.0 + 2.0 * part, rtol=1e-7)
    assert 0.0 <= full.min() and full.max() < 1.0 and abs(full.mean() - 0.5) < 0.01


@pytest.mark.parametrize("shape,r", [((64, 48, 128), 16), ((40, 24, 64), 40), ((6, 8, 16, 64), 9), ((130, 70, 192), 100), ((33, 8, 64), 5)])
def test_mttkrp_of_every_mode_in_place_over_one_copy_of_the_tensor(shape, r):
    """NMFPlan.view: the unfoldings of the modes >= 1 are TMA maps over the planes of unfold(T, 0) (MN-major operand for the last
    mode, 3-D map for middle modes) -- no unfolded copy (ntf.py:309-311).  MTTKRP of every mode against float64 numpy."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(sum(shape) + r)
    T = rng.rand(*shape).astype(np.float32)
    Td = torch.from_numpy(T).cuda()
    base = ops.NMFPlan(Td.reshape(shape[0], -1)).bind_rank(r, sides=1)
    nm = len(shape)
    for mode in range(nm):
        left, I, right = ops._split(list(shape), mode)
        plan = base if mode == 0 else base.view(left, I, right, r)
        assert plan is not None, (shape, mode)
        rest = int(np.prod(shape)) // shape[mode]
        Kt = rng.rand(r, rest).astype(np.float32)                      # any (r x rest) operand; NTF passes the Khatri-Rao product
        got = plan.cross(0, torch.from_numpy(Kt).cuda()).cpu().numpy()  # (unfold(T, mode) @ Kt^T)^T
        unf = np.moveaxis(T.astype(np.float64), mode, 0).reshape(shape[mode], -1)
        ref = Kt.astype(np.float64) @ unf.T
        np.testing.assert_allclose(got, ref, rtol=2e-5)
    # extents that cannot be addressed in place are refused, not mis-addressed
    odd = ops.NMFPlan(torch.rand((10, 6 * 50), device="cuda")).bind_rank(4, sides=1)
    assert odd.view(10, 6, 50, 4) is None                                 # padded planes (300 % 64 != 0)
    with pytest.raises(Exception):
        base.view(shape[0], int(np.prod(shape[1:])), 1, r).set_factor(0, torch.zeros((r, int(np.prod(shape[1:]))), device="cuda"))


# ---------------------------------------------------------------------------------------------
# BASELINE.json configs[1] at its FULL size (65536 x 8192, rank 64), through size-independent properties
# ---------------------------------------------------------------------------------------------
def _f64_costs_chunked(X, Ut, V, rows=4096):
    """||X - U V||^2 and KL(X | U V) in float64 with torch, 4096 rows of X at a time (an evaluation that shares nothing with
    the kernels under test)."""
    import torch
    fro = torch.zeros((), dtype=torch.float64, device=X.device)
    kl = torch.zeros((), dtype=torch.float64, device=X.device)
    V64 = V.double()
    for lo in range(0, X.shape[0], rows):
        x = X[lo:lo + rows].double()
        k = Ut[:, lo:lo + rows].double().T @ V64
        fro += ((x - k) ** 2).sum()
        kl += (x * torch.log(x / k) - x + k).sum()
    return float(fro), float(kl)


@pytest.mark.parametrize("rule", ["hals", "mu"])
def test_nmf_config2_full_size_against_oracle_on_subsamples(rule):
    """C2 (the headline configuration) at full size.  An update of U only couples the rows of U through the number of sweeps
    (nnls.py:156) and not at all for MU, so the float64 oracle restricted to a random subset of rows of X (columns for the V
    update), run for the sweep count the GPU reports, must reproduce those rows of the GPU result; the reported objective is
    checked against an independent float64 evaluation over the whole matrix, and must not increase."""
    import torch
    from nn_fac import _fast
    from oracle import nnfac_oracle as orc
    m, n, r = 65536, 8192, 64
    g = torch.Generator(device="cuda"); g.manual_seed(2024)
    W0, H0 = torch.rand((m, r), generator=g, device="cuda"), torch.rand((r, n), generator=g, device="cuda")
    X = W0 @ H0
    X += float(X.mean()) * torch.rand((m, n), generator=g, device="cuda") + 1e-3
    del W0, H0
    U0, V0 = torch.rand((m, r), generator=g, device="cuda"), torch.rand((r, n), generator=g, device="cuda")
    beta = 2 if rule == "hals" else 1
    assert _fast.eligible(torch.float32, r, rule, beta)
    st = _fast.FusedNMF(X, U0, V0)
    costs, _ = st.run(3, 0.0, rule, beta=beta)
    assert len(costs) == 3 and costs[0] >= costs[1] >= costs[2] > 0
    fro, kl = _f64_costs_chunked(X, st.Ut, st.V)
    want = fro if rule == "hals" else kl
    assert abs(costs[-1] - want) <= 1e-5 * want, (costs[-1], want)

    # one outer iteration from (U0, V0): rows of the new U, then columns of the new V, against the oracle on subsamples
    st = _fast.FusedNMF(X, U0, V0)
    st.run(1, 0.0, rule, beta=beta)
    U1t, V1 = st.Ut, st.V
    rs = np.random.RandomState(5)
    rows = torch.from_numpy(np.sort(rs.choice(m, 192, replace=False))).cuda()
    cols = torch.from_numpy(np.sort(rs.choice(n, 192, replace=False))).cuda()
    Xr, Xc = X[rows].double().cpu().numpy(), X[:, cols].double().cpu().numpy()
    U0r, V0c = U0[rows].double().cpu().numpy(), V0[:, cols].double().cpu().numpy()
    V0h, U1h = V0.double().cpu().numpy(), U1t.double().cpu().numpy().T
    if rule == "hals":
        cnt_U, cnt_V = [int(c) for c in st.sweep_log[0].cpu().tolist()]
        assert 2 <= cnt_U <= 100 and 2 <= cnt_V <= 100
        want_U = orc.hals_nnls_acc(V0h @ Xr.T, V0h @ V0h.T, U0r.T, maxiter=cnt_U, delta=0.0)[0].T      # nmf.py:407-416
        want_V = orc.hals_nnls_acc(U1h.T @ Xc, U1h.T @ U1h, V0c, maxiter=cnt_V, delta=0.0)[0]          # nmf.py:432-441
    else:
        want_U = orc.mu_betadivmin(U0r, V0h, Xr, 1)                                                    # mu.py:84-88
        want_V = orc.mu_betadivmin(V0c.T, U1h.T, Xc.T, 1).T                                            # mu.py:27
    got_U, got_V = U1h[rows.cpu().numpy()], V1[:, cols].double().cpu().numpy()
    assert np.linalg.norm(got_U - want_U) <= 2e-4 * np.linalg.norm(want_U)
    assert np.linalg.norm(got_V - want_V) <= 2e-4 * np.linalg.norm(want_V)
    assert (got_U >= 0).all() and (got_V >= 0).all()
