"""The CUDA-core layer against float64: the fp32 HALS sweeps, the strided split-K GEMM, the tensor helpers built on it and the
element-wise kernels.

This layer is the production path of the fp32x3 HALS solve, of fp32 solves with `normalize` / `nonzero` or more columns than the
tensor-core sweep keeps resident, of NTF-MU, NTD, PARAFAC2, the general-beta tensorial MU and the fp64 mode; it is also the
yardstick of the tensor-core tests that compare against "the generic path".  Everything here calls nn_fac._ops directly on device
tensors, so the routing of nn_fac.config plays no part.

Two kinds of check:
  * exact data -- small non-negative integers (0..3), wherever the operation allows it.  Every partial sum is then an integer
    below 2^24, so fp32 and fp64 results must equal float64 numpy bit for bit: one dropped, repeated or misplaced term fails;
  * random data against a stated rounding bound.  The worst error-to-bound ratio of every bounded test is collected and printed
    at the end of the module (run with -s to see it).

Which kernel, tiling and branch ran is predicted by helpers that restate the launch arithmetic of csrc/hals_sweep.cuh
(hals::launch / run_rank) and csrc/gemm_generic.cu (run_gemm) from the device's SM count, and the kernel names recorded by
torch.profiler are checked against those predictions.
"""
import numpy as np
import pytest

from oracle import nnfac_oracle as orc

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
U64 = 2.0 ** -53
_WORST = {}


def _record(name, ratio):
    _WORST[name] = max(_WORST.get(name, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    if _WORST:
        print("\nworst error / bound per test:")
        for k in sorted(_WORST):
            print(f"  {k:60s} {_WORST[k]:.3e}")


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    return t.cpu().numpy()


def _cdiv(a, b):
    return -(-a // b)


def _kernels(fn):
    """Names of the CUDA kernels `fn` launched (torch.profiler, CUDA activity).  A profiling session of a long-lived process now
    and then delivers no device activity at all (not even the copies every call makes); `fn` is deterministic, so such an empty
    capture is taken again."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        if names:
            return names
    raise AssertionError("the profiler recorded no CUDA activity in three captures")


def _ran(names, needle):
    return any(needle in n for n in names)


# =============================================================================================
# 1. fp32 CUDA-core HALS sweep
# =============================================================================================
# Tiling<float, RP> of csrc/hals_sweep.cuh: (WL, WC) lanes / columns of a group in the wide tiling, (NL, NC) in the narrow one
TILING32 = {16: (1, 4, 4, 1), 32: (1, 4, 8, 1), 64: (2, 4, 8, 1), 128: (4, 4, 16, 1)}


def sweep_plan(r, n, rowops, sms):
    """What nnfac_hals_nnls(fp32, NNFAC_HALS_NO_TC) launches: hals::run_rank / hals::launch restated."""
    if r > 128:
        return dict(tiling="general", kernel="gen_row_update_kernel<float>" if rowops else "gen_sweep_kernel<float>")
    rp = 16 if r <= 16 else 32 if r <= 32 else 64 if r <= 64 else 128
    wl, wc, nl, nc = TILING32[rp]
    if rowops:
        lanes, cols, maxt, tiling = wl, wc, 256, "rowops"
    else:
        wide_threads = _cdiv(n, wc) * wl
        narrow_fits = _cdiv(_cdiv(n, nc), sms) * nl <= 512
        if wide_threads >= sms * 128 or not narrow_fits:
            lanes, cols, maxt, tiling = wl, wc, 256, "wide"
        else:
            lanes, cols, maxt, tiling = nl, nc, 512, "narrow"
    groups = _cdiv(n, cols)
    grid = sms if groups * lanes >= sms * 32 else max(1, _cdiv(groups * lanes, 32))
    threads = _cdiv(_cdiv(groups, grid) * lanes, 32) * 32
    nbatch, per_batch = 1, None
    if threads > maxt:
        threads = maxt
        per_batch = (maxt // lanes) * cols * grid
        nbatch = _cdiv(n, per_batch)
    if rowops and nbatch > 1:
        return dict(tiling="general", kernel="gen_row_update_kernel<float>", rp=rp)
    smem_base = (rp * rp + rp) * 4 + 40 * 8
    slab = nbatch == 1 and smem_base + r * (threads // lanes) * cols * 4 <= 200 * 1024
    if rowops:
        kernel = f"hals_sweep_kernel<float, {rp}, {lanes}, {cols}, true, 256>"
    else:
        kernel = f"hals_sweep_chunked_kernel<float, {rp}, {lanes}, {cols}, {maxt}>"
    return dict(tiling=tiling, kernel=kernel, rp=rp, lanes=lanes, cols=cols, grid=grid, threads=threads, nbatch=nbatch,
                per_batch=per_batch, slab=slab)


def _first_n(pred, lo=1, hi=1 << 22):
    """Smallest n in [lo, hi] with pred(n) (pred monotone)."""
    assert pred(hi)
    while lo < hi:
        mid = (lo + hi) // 2
        if pred(mid):
            hi = mid
        else:
            lo = mid + 1
    return lo


def tiling_columns(rp, sms):
    """Column counts that reach every tiling of run_rank at padded rank rp: narrow from one column up to its limit, wide with
    one batch just past the switch and at its limit, and wide with three batches (ragged last batch and column group)."""
    r = rp
    n_sw = _first_n(lambda n: sweep_plan(r, n, False, sms)["tiling"] == "wide")
    wl, wc = TILING32[rp][:2]
    single_max = (256 // wl) * wc * sms
    return {"narrow": [1, 37, 1001, n_sw - 1], "wide1": [n_sw + 1, single_max - 3],
            "wideN": [2 * single_max + single_max // 3 + 1]}


def _nnls_problem(r, n, seed):
    """fp32 UtM (r x n), UtU (r x r), V0 (r x n) of a least-squares problem min ||M - U V|| with m = 2r + 8 rows, a sparse
    non-negative solution and noise (so that the solution has active bounds)."""
    rng = np.random.RandomState(seed)
    m = 2 * r + 8
    U = rng.rand(m, r) + 0.05
    G = U.T @ U
    Vt = rng.rand(r, n) * (rng.rand(r, n) > 0.3)
    UtM = G @ Vt + 0.3 * np.sqrt(m) * rng.randn(r, n)
    V0 = rng.rand(r, n)
    return UtM.astype(np.float32), G.astype(np.float32), V0.astype(np.float32)


def _run_sweep(UtM, UtU, V0, r, maxiter, delta, sp=0.0, normalize=False, nonzero=False):
    from nn_fac import _ops as ops
    b, G, V = _dev(UtM), _dev(UtU), _dev(V0)
    res = ops.hals_nnls(b, G, V, r, int(maxiter), delta, sp, normalize, nonzero, no_tc=True)
    return _host(V), _host(res)


# Acceptance of a whole solve (docstring of test_sweep_padded_ranks): relative Frobenius error of V and relative error of eps
REL_V = 2e-5
REL_EPS = 5e-5


def _check_solve(name, UtM, UtU, V0, r, maxiter, delta, sp=0.0, normalize=False, nonzero=False):
    V, res = _run_sweep(UtM, UtU, V0, r, maxiter, delta, sp, normalize, nonzero)
    f = lambda x: x.astype(np.float64)  # noqa: E731
    Vo, eps_o, cnt_o, _ = orc.hals_nnls_acc(f(UtM), f(UtU), f(V0), maxiter=maxiter, delta=delta,
                                            sparsity_coefficient=sp or None, normalize=normalize, nonzero=nonzero)
    assert res[2] == -1.0
    assert abs(int(res[1]) - cnt_o) <= 1, (name, res[1], cnt_o)
    assert res[3] == res[1] - 1
    assert np.all(V >= 0) and np.all(np.isfinite(V))
    if int(res[1]) == cnt_o:
        ev = np.linalg.norm(V - Vo) / max(np.linalg.norm(Vo), 1e-300)
        # a solve that has converged sweeps steps of rounding size: eps is then noise, at most a rounding-level step
        # (r + 2) 2^-24 max|V| in every entry, squared and summed
        floor = Vo.size * ((r + 2) * U32 * np.abs(Vo).max()) ** 2
        ee = abs(res[0] - eps_o) / (REL_EPS * abs(eps_o) + floor)
        _record(name + " V", ev / REL_V)
        _record(name + " eps", ee)
        assert ev <= REL_V, (name, ev)
        assert ee <= 1.0, (name, res[0], eps_o, floor)
    return V, res


RANKS = [1, 5, 16, 17, 32, 33, 64, 65, 100, 128]


@pytest.mark.parametrize("r", RANKS)
def test_sweep_padded_ranks(r, sms):
    """Every padded rank RP in {16, 32, 64, 128}, at ranks on both sides of each padding boundary, on the narrow tiling (n = 1001)
    and the wide one (n just past the switch), 8 sweeps at delta = 0 and a delta-stopped solve.

    Bound: the fp32 sweep is plain FMA arithmetic, so its result differs from the float64 sweep by rounding amplified through a
    few Gauss-Seidel sweeps.  The bounds are a relative Frobenius error of V of REL_V = 2e-5 (about 340 units of 2^-24) and a
    relative error of eps (the sum of squared steps of the last sweep) of REL_EPS = 5e-5.  A converged solve (r = 1 is solved by
    its first sweep) sweeps rounding-size steps, so eps also gets an absolute floor of a (r + 2) 2^-24 max|V| step in every
    entry.  Measured on a B200 (148 SMs) over every solve of this module, the worst errors were 7.8e-6 for V (0.39 of REL_V) and
    8e-6 for eps (0.17 of REL_EPS): much tighter than the 5e-4 of the tensor-core sweep, which splits operands into bf16."""
    rp = sweep_plan(r, 1001, False, sms)["rp"]
    n_wide = tiling_columns(rp, sms)["wide1"][0]
    for n in (1001, n_wide):
        UtM, UtU, V0 = _nnls_problem(r, n, 100 * r + n % 97)
        _check_solve("padded ranks", UtM, UtU, V0, r, 8, 0.0)
    UtM, UtU, V0 = _nnls_problem(r, 1001, r + 5)
    _check_solve("padded ranks, delta stop", UtM, UtU, V0, r, 200, 0.01)


@pytest.mark.parametrize("kind", ["narrow", "wide1", "wideN"])
@pytest.mark.parametrize("rp", [16, 32, 64, 128])
def test_sweep_every_tiling(rp, kind, sms):
    """Every tiling of run_rank at every padded rank: narrow (NL lanes, 512 threads) from one column up to its limit, wide with
    one batch (UtM slab in shared memory), and wide with three batches (no slab; ragged last batch and last column group).
    Rank RP - 3 or RP // 2 + 1 (a padded rank with zero rows).  Bounds as in test_sweep_padded_ranks."""
    r = {16: 13, 32: 29, 64: 50, 128: 100}[rp]
    for n in tiling_columns(rp, sms)[kind]:
        p = sweep_plan(r, n, False, sms)
        assert p["rp"] == rp and p["tiling"] == ("narrow" if kind == "narrow" else "wide"), (n, p)
        if kind == "wideN":
            assert p["nbatch"] == 3 and not p["slab"] and n % p["per_batch"] != 0 and n % p["cols"] != 0, p
        else:
            assert p["nbatch"] == 1 and p["slab"], p
        UtM, UtU, V0 = _nnls_problem(r, n, rp + n)
        _check_solve(f"tiling {kind}", UtM, UtU, V0, r, 2 if n > 50000 else 5, 0.0)


def test_sweep_narrow_wide_switch_on_both_sides(sms):
    """The same column count at two ranks, narrow at RP = 64 and wide at RP = 128."""
    n = tiling_columns(128, sms)["wide1"][0]
    assert sweep_plan(60, n, False, sms)["tiling"] == "narrow" and sweep_plan(120, n, False, sms)["tiling"] == "wide"
    for r in (60, 120):
        UtM, UtU, V0 = _nnls_problem(r, n, r)
        _check_solve("switch", UtM, UtU, V0, r, 5, 0.0)


def _single_sweep_bound(UtM, UtU, V0, sp):
    """Element-wise rounding bound of one fp32 sweep, evaluated in float64 along the oracle's sweep.  Row k is
    d = max((b_k - G_k. v - sp) / G_kk, -v_k): an (r + 2)-term computation whose rounding is at most
    2^-24 (r + 2) (|b_k| + sp + sum_j |G_kj| (|V0_j| + |V_j|)) / G_kk (the chunked kernel forms G_kj V_j of the rows already updated
    in the chunk as G_kj V0_j + G_kj d_j, hence both values of V_j), plus the propagated error sum_{j<k} |G_kj| err_j / G_kk of the
    rows updated before it.  kappa = 1."""
    b, G, V = (x.astype(np.float64) for x in (UtM, UtU, V0))
    V0d = V.copy()
    r = b.shape[0]
    err = np.zeros_like(V)
    for k in range(r):
        if G[k, k] == 0:
            continue
        scale = (np.abs(b[k]) + abs(sp) + np.abs(G[k]) @ (np.abs(V0d) + np.abs(V))) / G[k, k]
        prop = np.abs(G[k]) @ err / G[k, k]
        step = np.maximum((b[k] - G[k] @ V - sp) / G[k, k], -V[k])
        V[k] += step
        err[k] = (r + 2) * U32 * scale + prop
    return V, err


@pytest.mark.parametrize("r,n", [(1, 5), (16, 1001), (17, 333), (64, 4000), (100, 3001), (128, 50000), (160, 700)])
@pytest.mark.parametrize("sp", [0.0, 0.4])
def test_single_sweep_elementwise(r, n, sp, sms):
    """maxiter = 1 element by element against the oracle's single sweep, within the bound of _single_sweep_bound (kappa = 1):
    narrow, wide, the general sweep (r = 160), with and without sparsity."""
    UtM, UtU, V0 = _nnls_problem(r, n, r * 3 + n)
    V, res = _run_sweep(UtM, UtU, V0, r, 1, 0.01, sp)
    Vo, bound = _single_sweep_bound(UtM, UtU, V0, sp)
    Vr, _, cnt_o, _ = orc.hals_nnls_acc(UtM.astype(np.float64), UtU.astype(np.float64), V0.astype(np.float64), maxiter=1,
                                        sparsity_coefficient=sp or None)
    np.testing.assert_allclose(Vo, Vr, rtol=1e-12, atol=1e-12)
    assert int(res[1]) == cnt_o == 2
    ratio = np.abs(V - Vo) / np.maximum(bound, 1e-300)
    _record("single sweep elementwise", ratio.max())
    assert ratio.max() <= 1.0, (np.unravel_index(ratio.argmax(), ratio.shape), ratio.max())


OPTS = {"normalize": dict(normalize=True), "nonzero": dict(nonzero=True), "both": dict(normalize=True, nonzero=True)}


@pytest.mark.parametrize("sp", [0.0, 0.3])
@pytest.mark.parametrize("opt", sorted(OPTS))
@pytest.mark.parametrize("r,n", [(5, 300), (16, 4001), (33, 1000), (100, 2500)])
def test_sweep_row_operations(r, n, opt, sp, sms):
    """The ROWOPS kernel (the only kernel for normalize / nonzero while all columns are resident) against the oracle."""
    assert sweep_plan(r, n, True, sms)["tiling"] == "rowops"
    UtM, UtU, V0 = _nnls_problem(r, n, r + n + len(opt))
    _check_solve(f"rowops {opt}", UtM, UtU, V0, r, 6, 0.0, sp=sp, **OPTS[opt])
    _check_solve(f"rowops {opt} delta", UtM, UtU, V0, r, 60, 0.01, sp=sp, **OPTS[opt])


@pytest.mark.parametrize("opt", ["nonzero", "both"])
@pytest.mark.parametrize("r,n,tiling", [(16, 1000, "rowops"), (64, 2000, "rowops"), (150, 600, "general"),
                                        (16, None, "general")])
def test_sweep_row_driven_to_zero_is_refilled(r, n, tiling, opt, sms):
    """A row whose right-hand side is negative everywhere is driven to zero by the first sweep; with `nonzero` it is refilled with
    1e-16 max(V) (nnls.py:173-174), on the ROWOPS kernel and on the general sweep (also in fp32 past the resident limit).  After one
    sweep the refilled row must equal the oracle's within 1e-5 relative: max(V) carries the fp32 error of the rows already swept
    (about 1e-6) and the fill one rounding, so a fill of the wrong scale (1e-15 max(V), say) fails; with `normalize` as well the
    row is 1 / sqrt(n)."""
    if n is None:
        n = _first_n(lambda k: sweep_plan(16, k, True, sms)["tiling"] == "general")
    assert sweep_plan(r, n, True, sms)["tiling"] == tiling
    UtM, UtU, V0 = _nnls_problem(r, n, r + n)
    UtM[3] = -50.0 * np.abs(UtM[3]) - 1.0
    V, res = _check_solve(f"refill {tiling}", UtM, UtU, V0, r, 3, 0.0, **OPTS[opt])
    Vo, _, _, _ = orc.hals_nnls_acc(UtM.astype(np.float64), UtU.astype(np.float64), V0.astype(np.float64), maxiter=1,
                                    **OPTS[opt])
    assert np.all(Vo[3] > 0) and np.ptp(Vo[3]) == 0
    assert np.all(V[3] > 0)
    V1, _ = _run_sweep(UtM, UtU, V0, r, 1, 0.0, **OPTS[opt])
    np.testing.assert_allclose(V1[3], Vo[3], rtol=1e-5, atol=0)


@pytest.mark.parametrize("r,n", [(20, 500), (100, 3000), (140, 300), (16, None)])
def test_sweep_zero_diagonal(r, n, sms):
    """A zero diagonal entry of UtU: the row is skipped (plain, sparsity, normalize), and with `nonzero` the solve stops with that
    row in result[2] (ZeroColumnWhenUnautorized in nnls.py)."""
    if n is None:
        n = _first_n(lambda k: sweep_plan(16, k, True, sms)["tiling"] == "general") + 7
    UtM, UtU, V0 = _nnls_problem(r, n, r + n)
    k = r // 2 + 1
    UtU[k, :] = 0
    UtU[:, k] = 0
    for kw in ({}, dict(sp=0.2), dict(normalize=True)):
        V, _ = _check_solve("zero diagonal", UtM, UtU, V0, r, 4, 0.0, **kw)
        if not kw.get("normalize"):
            np.testing.assert_array_equal(V[k], V0[k])
    for kw in (dict(nonzero=True), dict(nonzero=True, normalize=True)):
        _, res = _run_sweep(UtM, UtU, V0, r, 4, 0.0, **kw)
        assert res[2] == k
        with pytest.raises(ZeroDivisionError):
            orc.hals_nnls_acc(UtM.astype(np.float64), UtU.astype(np.float64), V0.astype(np.float64), maxiter=4, **kw)


@pytest.mark.parametrize("opt", ["normalize", "nonzero"])
def test_sweep_row_operations_past_the_resident_columns_go_to_the_general_sweep(opt, sms):
    """fp32 normalize / nonzero on more columns than the ROWOPS kernel keeps resident run the general sweep; the kernel that ran is
    the general row kernel."""
    n = _first_n(lambda k: sweep_plan(16, k, True, sms)["tiling"] == "general") + 11
    r = 16
    UtM, UtU, V0 = _nnls_problem(r, n, 7)
    names = _kernels(lambda: _run_sweep(UtM, UtU, V0, r, 1, 0.0, **OPTS[opt]))
    assert _ran(names, "gen_row_update_kernel<float>") and not _ran(names, "hals_sweep_kernel")
    _check_solve("rowops general", UtM, UtU, V0, r, 3, 0.0, **OPTS[opt])


@pytest.mark.parametrize("r", [129, 160])
@pytest.mark.parametrize("opt", ["plain", "sparsity", "normalize", "nonzero", "both"])
def test_general_sweep_fp32(r, opt):
    kw = {"plain": {}, "sparsity": dict(sp=0.5)}.get(opt, OPTS.get(opt, {}))
    UtM, UtU, V0 = _nnls_problem(r, 777, r)
    _check_solve("general", UtM, UtU, V0, r, 6, 0.0, **kw)
    _check_solve("general delta", UtM, UtU, V0, r, 60, 0.01, **kw)


@pytest.mark.parametrize("opt", ["plain", "normalize"])
@pytest.mark.parametrize("r,n", [(13, 1001), (50, 6000), (100, 40001), (150, 500)])
def test_sweep_strided_operands(r, n, opt):
    """UtM, UtU and V as column slices of wider buffers (ld > n) whose other columns hold NaN: the NaN is never read (the result
    equals the contiguous solve bit for bit) and never overwritten.  Two offsets: 16-byte aligned and not."""
    import torch
    from nn_fac import _ops as ops
    kw = OPTS.get(opt, {})
    UtM, UtU, V0 = _nnls_problem(r, n, r + n)
    Vc, resc = _run_sweep(UtM, UtU, V0, r, 4, 0.0, **kw)
    for off in (4, 3):
        ld = n + off + 5
        bb = torch.full((r, ld), float("nan"), device="cuda")
        vb = torch.full((r, ld), float("nan"), device="cuda")
        gb = torch.full((r, r + 3), float("nan"), device="cuda")
        bb[:, off:off + n] = _dev(UtM)
        vb[:, off:off + n] = _dev(V0)
        gb[:, :r] = _dev(UtU)
        res = ops.hals_nnls(bb[:, off:off + n], gb[:, :r], vb[:, off:off + n], r, 4, 0.0, 0.0, kw.get("normalize", False),
                            False, no_tc=True)
        vh = _host(vb)
        np.testing.assert_array_equal(vh[:, off:off + n], Vc)
        np.testing.assert_array_equal(_host(res), resc)
        assert np.isnan(vh[:, :off]).all() and np.isnan(vh[:, off + n:]).all()
        assert np.isnan(_host(bb)[:, :off]).all() and np.isnan(_host(gb)[:, r:]).all()
        np.testing.assert_array_equal(_host(bb)[:, off:off + n], UtM)
    _check_solve("strided", UtM, UtU, V0, r, 4, 0.0, **kw)


@pytest.mark.parametrize("r,n", [(5, 300), (64, 3000), (100, 40001), (150, 400)])
def test_sweep_iteration_edges(r, n):
    """maxiter 0 (V untouched, eps = 1, cnt = 1), 1 and 2; delta = 0 runs to maxiter; a zero right-hand side from V = 0 moves
    nothing, and the reference then counts all maxiter sweeps (cnt = maxiter + 1)."""
    UtM, UtU, V0 = _nnls_problem(r, n, n)
    V, res = _run_sweep(UtM, UtU, V0, r, 0, 0.01)
    np.testing.assert_array_equal(V, V0)
    assert list(res[:3]) == [1.0, 1.0, -1.0]
    for opt in ({}, dict(normalize=True)):
        for maxiter in (1, 2):
            _, res = _check_solve("iteration edges", UtM, UtU, V0, r, maxiter, 0.01, **opt)
            assert res[1] == maxiter + 1
        _, res = _check_solve("iteration edges", UtM, UtU, V0, r, 7, 0.0, **opt)
        assert res[1] == 8
    Z = np.zeros_like(V0)
    V, res = _run_sweep(Z, UtU, Z, r, 9, 0.01)
    _, eps_o, cnt_o, _ = orc.hals_nnls_acc(Z.astype(np.float64), UtU.astype(np.float64), Z.astype(np.float64), maxiter=9)
    assert not V.any() and res[0] == eps_o == 0.0 and res[1] == cnt_o == 10


@pytest.mark.parametrize("opt", ["plain", "normalize", "nonzero"])
@pytest.mark.parametrize("r,n", [(16, 1001), (64, 100001), (100, 3001), (140, 500)])
def test_sweep_reruns_are_bit_identical(r, n, opt):
    UtM, UtU, V0 = _nnls_problem(r, n, 3)
    kw = OPTS.get(opt, {})
    runs = [_run_sweep(UtM, UtU, V0, r, 5, 0.01, sp=0.1, **kw) for _ in range(3)]
    for V, res in runs[1:]:
        np.testing.assert_array_equal(V, runs[0][0])
        np.testing.assert_array_equal(res, runs[0][1])


def test_sweep_kernel_names_match_the_launch_arithmetic(sms):
    """The kernel torch.profiler records for every tiling, padded rank and option is the one sweep_plan predicts."""
    seen = []
    for rp, r in ((16, 13), (32, 29), (64, 50), (128, 100)):
        cols = tiling_columns(rp, sms)
        for n in (cols["narrow"][2], cols["wide1"][0], cols["wideN"][0]):
            for rowops in (False, True):
                p = sweep_plan(r, n, rowops, sms)
                UtM, UtU, V0 = _nnls_problem(r, n, 1)
                names = _kernels(lambda: _run_sweep(UtM, UtU, V0, r, 1, 0.0, normalize=rowops))
                assert _ran(names, p["kernel"]), (r, n, rowops, p, sorted(set(names)))
                assert not _ran(names, "tc_sweep"), names
                seen.append((r, n, rowops, p["tiling"], p.get("nbatch"), p.get("slab"), p["kernel"]))
    for r in (129, 160):
        UtM, UtU, V0 = _nnls_problem(r, 300, 1)
        names = _kernels(lambda: _run_sweep(UtM, UtU, V0, r, 1, 0.0))
        assert _ran(names, "gen_sweep_kernel<float>")
        seen.append((r, 300, False, "general", None, None, "gen_sweep_kernel<float>"))
    print("\nsweep routing (r, n, rowops, tiling, nbatch, slab, kernel):")
    for s in seen:
        print("  ", s)


# =============================================================================================
# 2. strided / batched / split-K GEMM
# =============================================================================================
def gemm_plan(M, N, K, kb, batch, sms):
    """run_gemm's split-K choice (csrc/gemm_generic.cu) restated."""
    kbq = _cdiv(K, 16)
    nblk = kb * kbq
    tiles = _cdiv(M, 64) * _cdiv(N, 64) * batch
    splits = 1
    capped = False
    if tiles < 2 * sms:
        splits = _cdiv(2 * sms, tiles)
        splits = min(splits, max(nblk // 8, 1))
        capped = splits > 256
        splits = min(splits, 256)
    bps = _cdiv(nblk, splits)
    splits = _cdiv(nblk, bps)
    return dict(splits=splits, bps=bps, nblk=nblk, kbq=kbq, capped=capped, last=nblk - (splits - 1) * bps)


def _extent(shape, strides):
    return 1 + sum((s - 1) * abs(st) for s, st in zip(shape, strides))


def _layout(M, N, K, kb, batch, a_kcontig, b_jcontig, pad=3):
    """Strides (elements) of A and B: the four load paths of gemm_strided_kernel, padded leading dimensions, q- and batch-blocks
    with gaps."""
    if a_kcontig:
        sa_i, sa_k = K + pad, 1
    else:
        sa_i, sa_k = 1, M + pad
    sa_q = _extent((M, K), (sa_i, sa_k)) + pad
    sa_b = kb * sa_q + 2 * pad
    if b_jcontig:
        sb_k, sb_j = N + pad, 1
    else:
        sb_k, sb_j = 1, K + pad
    sb_q = _extent((K, N), (sb_k, sb_j)) + pad
    sb_b = kb * sb_q + 5
    return (sa_i, sa_k, sa_q, sa_b), (sb_k, sb_j, sb_q, sb_b)


def _strided_ref(Ah, a_str, Bh, b_str, M, N, K, kb, batch):
    """C[b,i,j] = sum_q sum_k A[b sa_b + q sa_q + i sa_i + k sa_k] B[b sb_b + q sb_q + k sb_k + j sb_j] in float64, and the same
    with |A|, |B|."""
    from numpy.lib.stride_tricks import as_strided
    sa_i, sa_k, sa_q, sa_b = a_str
    sb_k, sb_j, sb_q, sb_b = b_str
    A64, B64 = Ah.astype(np.float64), Bh.astype(np.float64)
    e = 8
    Av = as_strided(A64, (batch, kb, M, K), (sa_b * e, sa_q * e, sa_i * e, sa_k * e), writeable=False)
    Bv = as_strided(B64, (batch, kb, K, N), (sb_b * e, sb_q * e, sb_k * e, sb_j * e), writeable=False)
    C = np.zeros((batch, M, N))
    Cabs = np.zeros((batch, M, N))
    for q in range(kb):
        C += np.matmul(Av[:, q], Bv[:, q])
        Cabs += np.matmul(np.abs(Av[:, q]), np.abs(Bv[:, q]))
    return C, Cabs


def _data(size, kind, dtype, rng):
    if kind == "exact":
        return rng.randint(0, 4, size).astype(dtype)
    return rng.uniform(-1, 1, size).astype(dtype)


def _check_gemm(name, M, N, K, kb, batch, a_kcontig, b_jcontig, dtype, kind, sms, out_gaps=False, rng=None):
    import torch
    from nn_fac import _ops as ops
    rng = rng or np.random.RandomState(M * 7 + N * 3 + K + kb)
    a_str, b_str = _layout(M, N, K, kb, batch, a_kcontig, b_jcontig)
    Ah = _data(_extent((batch, kb, M, K), (a_str[3], a_str[2], a_str[0], a_str[1])), kind, dtype, rng)
    Bh = _data(_extent((batch, kb, K, N), (b_str[3], b_str[2], b_str[0], b_str[1])), kind, dtype, rng)
    A, B = _dev(Ah), _dev(Bh)
    if out_gaps:
        ldc, sc_b = N + 5, (N + 5) * M + 7
        buf = torch.full((_extent((batch, M, N), (sc_b, ldc, 1)) + 9,), float("nan"), dtype=A.dtype, device="cuda")
        ops.gemm(A, a_str, B, b_str, M, N, K, kb=kb, batch=batch, out=buf, ldc=ldc, sc_b=sc_b)
        h = _host(buf)
        mask = np.zeros(h.shape, bool)
        idx = (np.arange(batch)[:, None, None] * sc_b + np.arange(M)[None, :, None] * ldc + np.arange(N)[None, None, :]).ravel()
        mask[idx] = True
        assert np.isnan(h[~mask]).all(), name
        C = h[idx].reshape(batch, M, N)
    else:
        C = _host(ops.gemm(A, a_str, B, b_str, M, N, K, kb=kb, batch=batch)).reshape(batch, M, N)
    C64, Cabs = _strided_ref(Ah, a_str, Bh, b_str, M, N, K, kb, batch)
    if kind == "exact":
        assert Cabs.max() < 2 ** 24
        np.testing.assert_array_equal(C, C64, err_msg=name)
    else:
        p = gemm_plan(M, N, K, kb, batch, sms)
        chain = min(p["bps"] * 16, K * kb) + p["splits"]
        if dtype == np.float32:
            bound = chain * U32 * Cabs
        else:                                   # the float64 reference rounds too: its own K kb-term sums
            bound = (chain + K * kb) * U64 * Cabs
        ratio = (np.abs(C - C64) / np.maximum(bound, 1e-300)).max()
        _record(name, ratio)
        assert ratio <= 1.0, (name, ratio)
    return C


GEMM_MN = [(1, 1), (63, 65), (64, 64), (65, 63), (130, 130), (1, 130), (130, 1), (65, 1)]
GEMM_K = [1, 15, 16, 17, 1000]


@pytest.mark.parametrize("kind", ["exact", "random"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("a_kcontig,b_jcontig", [(True, True), (True, False), (False, True), (False, False)])
def test_gemm_load_paths_and_ragged_tiles(a_kcontig, b_jcontig, dtype, kind, sms):
    """All four load paths (sa_k == 1 or not x sb_j == 1 or not) at ragged M, N in {1, 63, 64, 65, 130} and K in
    {1, 15, 16, 17, 1000, 100003}, kb = 1 and kb = 3 (the zero-filled K tail of every q-block when K % 16 != 0).
    Random-data bound: |C - C64| <= kappa 2^-24 (min(16 bps, K kb) + splits) (|A||B|)_ij in fp32 (one FMA chain per split, then
    the fixed-order sum of the splits), kappa = 1; in fp64 2^-53 and the float64 reference's own K kb-term chain added."""
    name = f"gemm load paths {np.dtype(dtype).name} {kind}"
    for M, N in GEMM_MN:
        for K in GEMM_K:
            for kb in (1, 3):
                _check_gemm(name, M, N, K, kb, 1, a_kcontig, b_jcontig, dtype, kind, sms)
    for M, N in ((1, 1), (65, 1), (1, 63), (17, 33)):
        _check_gemm(name, M, N, 100003, 1, 1, a_kcontig, b_jcontig, dtype, kind, sms)


SPLIT_CASES = {
    # name: (M, N, K, kb, batch)
    "short last split": (64, 64, 4000, 1, 1),
    "boundaries inside q-blocks": (40, 50, 900, 3, 1),
    "256 cap": (1, 1, 100003, 1, 1),
    "batch x splits": (65, 63, 5003, 1, 3),
    "kb x batch x splits": (30, 70, 333, 7, 2),
    "no split": (130, 130, 1000, 2, 33),
}


@pytest.mark.parametrize("case", sorted(SPLIT_CASES))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gemm_split_k(case, dtype, sms):
    """Split-K: few tiles and long K, a short last split, split boundaries inside a q-block, the 256 cap, batch > 1 with splits > 1,
    each also into a strided output (ldc > N, sc_b > M N) whose gaps hold NaN that must survive.  Exact data bit for bit, random
    data within the bound of test_gemm_load_paths_and_ragged_tiles.  The kernels that ran are checked with the profiler."""
    M, N, K, kb, batch = SPLIT_CASES[case]
    p = gemm_plan(M, N, K, kb, batch, sms)
    if case == "no split":
        assert p["splits"] == 1
    else:
        assert p["splits"] > 1
    if case == "short last split":
        assert p["last"] < p["bps"]
    if case == "boundaries inside q-blocks":
        assert any((s * p["bps"]) % p["kbq"] for s in range(1, p["splits"])) and K % 16
    if case == "256 cap" and sms * 2 > 256:
        assert p["capped"] and p["last"] < p["bps"]
    for a_kc, b_jc in ((True, True), (False, False)):
        for kind in ("exact", "random"):
            for gaps in (False, True):
                _check_gemm(f"gemm split-K {np.dtype(dtype).name} {kind}", M, N, K, kb, batch, a_kc, b_jc, dtype, kind, sms,
                            out_gaps=gaps)
    names = _kernels(lambda: _check_gemm("profiled", M, N, K, kb, batch, True, True, dtype, "exact", sms))
    tn = "float" if dtype == np.float32 else "double"
    assert _ran(names, f"gemm_strided_kernel<{tn}>")
    assert _ran(names, f"splitk_reduce_kernel<{tn}>") == (p["splits"] > 1), (p, sorted(set(names)))


def test_gemm_stride_zero_operands():
    """Stride-0 operands: a one-element ones marker (strides (0, 0, 0, 0)) and a B shared by every batch (sb_b = 0)."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(0)
    Bh = rng.randint(0, 4, (37, 1001)).astype(np.float32)
    one = torch.ones(1, device="cuda")
    C = _host(ops.gemm(one, (0, 0, 0, 0), _dev(Bh), (1001, 1, 0, 0), 1, 1001, 37))
    np.testing.assert_array_equal(C.ravel(), Bh.astype(np.float64).sum(0))
    Ah = rng.randint(0, 4, (5, 40, 70)).astype(np.float32)
    Bs = rng.randint(0, 4, (70, 33)).astype(np.float32)
    C = _host(ops.gemm(_dev(Ah), (70, 1, 0, 40 * 70), _dev(Bs), (33, 1, 0, 0), 40, 33, 70, batch=5))
    np.testing.assert_array_equal(C, Ah.astype(np.float64) @ Bs.astype(np.float64))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gemm_reruns_bit_identical_on_two_streams(dtype, sms):
    """Split and unsplit products rerun bit for bit, on the same stream and on a second stream (the workspace guard)."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(1)
    for M, N, K, kb, batch in ((64, 64, 4000, 1, 1), (65, 63, 5003, 1, 3), (130, 130, 1000, 2, 9)):
        a_str, b_str = _layout(M, N, K, kb, batch, True, False)
        A = _dev(_data(_extent((batch, kb, M, K), (a_str[3], a_str[2], a_str[0], a_str[1])), "random", dtype, rng))
        B = _dev(_data(_extent((batch, kb, K, N), (b_str[3], b_str[2], b_str[0], b_str[1])), "random", dtype, rng))
        ref = _host(ops.gemm(A, a_str, B, b_str, M, N, K, kb=kb, batch=batch))
        np.testing.assert_array_equal(_host(ops.gemm(A, a_str, B, b_str, M, N, K, kb=kb, batch=batch)), ref)
        s2 = torch.cuda.Stream()
        s2.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s2):
            C2 = ops.gemm(A, a_str, B, b_str, M, N, K, kb=kb, batch=batch)
        torch.cuda.current_stream().wait_stream(s2)
        np.testing.assert_array_equal(_host(C2), ref)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("r", [1, 17, 64, 65, 100, 128, 130])
def test_gram_exact(r, dtype, sms):
    """F F^T on exact data, bit for bit: gram_partial_kernel (r <= 64), gram2_partial_kernel (64 < r <= 128, fp32) and the general
    GEMM beyond, at lengths that leave a ragged last CTA range and a ragged last slab, from a strided F (ld > len)."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(r)
    for length in (1, 63, 4 * sms * 64 + 17, 300007):
        Fh = rng.randint(0, 4, (r, length + 3)).astype(dtype)
        F = _dev(Fh)[:, :length]
        G = _host(ops.gram(F))
        F64 = Fh[:, :length].astype(np.float64)
        np.testing.assert_array_equal(G, F64 @ F64.T)


# =============================================================================================
# 3. tensor helpers on the GEMM
# =============================================================================================
def _ints(shape, rng, dtype, lo=0, hi=4):
    return rng.randint(lo, hi, shape).astype(dtype)


SHAPES3 = [(7, 65, 3), (1, 130, 17), (33, 5, 64)]
SHAPES4 = [(3, 5, 7, 9), (2, 17, 1, 66)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES3 + SHAPES4 + [(20000, 3, 5)])
def test_mode_dot_every_mode(shape, dtype):
    """mode_dot of every mode, plain and transposed, against numpy on exact data: right == 1 (the last mode), the batched branch,
    and its chunk loop (left > 16384, shape (20000, 3, 5) in mode 1)."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(len(shape))
    T = _ints(shape, rng, dtype)
    Td = _dev(T)
    for mode in range(len(shape)):
        R = 1 + (shape[mode] * 3) % 11
        M = _ints((R, shape[mode]), rng, dtype)
        ref = orc.mode_dot(T.astype(np.float64), M.astype(np.float64), mode)
        np.testing.assert_array_equal(_host(ops.mode_dot(Td, _dev(M), mode)), ref)
        np.testing.assert_array_equal(_host(ops.mode_dot(Td, _dev(np.ascontiguousarray(M.T)), mode, transpose=True)), ref)


@pytest.mark.parametrize("shape", SHAPES3 + SHAPES4)
def test_multi_mode_dot_with_skip(shape):
    from nn_fac import _ops as ops
    rng = np.random.RandomState(3)
    T = _ints(shape, rng, np.float64)
    mats = [_ints((1 + (s * 5) % 7, s), rng, np.float64) for s in shape]
    for skip in [None] + list(range(len(shape))):
        ref = orc.multi_mode_dot(T, mats, skip=skip)
        np.testing.assert_array_equal(_host(ops.multi_mode_dot(_dev(T), [_dev(m) for m in mats], skip=skip)), ref)
        refT = orc.multi_mode_dot(T, [m.T for m in mats], skip=skip, transpose=True)
        got = ops.multi_mode_dot(_dev(T), [_dev(np.ascontiguousarray(m.T)) for m in mats], skip=skip, transpose=True)
        np.testing.assert_array_equal(_host(got), refT)
    T32 = T.astype(np.float32)
    ref = orc.multi_mode_dot(T32.astype(np.float64), [m.astype(np.float64) for m in mats])
    assert np.abs(ref).max() < 2 ** 24
    np.testing.assert_array_equal(_host(ops.multi_mode_dot(_dev(T32), [_dev(m.astype(np.float32)) for m in mats])), ref)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", SHAPES3 + SHAPES4 + [(300, 40, 7)])
def test_unfold_times_every_mode(shape, dtype):
    """unfold(P, mode) @ unfold(B, mode)^T: the right == 1 branch (last mode), the kb branch (every other mode) and the 0-d ones
    marker (row sums of the unfolding)."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(11)
    B = _ints(shape, rng, dtype)
    for mode in range(len(shape)):
        pshape = list(shape)
        pshape[mode] = 1 + (shape[mode] * 7) % 13
        P = _ints(pshape, rng, dtype)
        ref = orc.unfold(P.astype(np.float64), mode) @ orc.unfold(B.astype(np.float64), mode).T
        np.testing.assert_array_equal(_host(ops.unfold_times(_dev(P), _dev(B), mode)), ref)
        one = torch.ones((), dtype=_dev(B).dtype, device="cuda")
        np.testing.assert_array_equal(_host(ops.unfold_times(one, _dev(B), mode)), orc.unfold(B.astype(np.float64), mode).sum(1))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_khatri_rao_transpose_and_small_kernels(dtype, sms):
    """khatri_rao against oracle.khatri_rao, transpose with ragged 32-tiles, hadamard_ and axpby, all bit for bit on exact data;
    norm1 on signed data; normalize_rows_ (a zero row stays zero) within 4 units of the format."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(5)
    for I, J, r in ((1, 1, 1), (7, 33, 5), (130, 65, 64), (1000, 3, 130)):
        A, B = _ints((I, r), rng, dtype), _ints((J, r), rng, dtype)
        np.testing.assert_array_equal(_host(ops.khatri_rao(_dev(A), _dev(B))), orc.khatri_rao([A, B]))
    for rows, cols in ((1, 1), (31, 33), (32, 32), (65, 1), (1, 100), (1000, 97)):
        X = _ints((rows, cols + 3), rng, dtype, -9, 9)
        np.testing.assert_array_equal(_host(ops.transpose(_dev(X)[:, :cols])), X[:, :cols].T)
    for count in (1, 1000, 256 * sms * 16 + 13):
        X, Y = _ints(count, rng, dtype, -9, 9), _ints(count, rng, dtype, -9, 9)
        np.testing.assert_array_equal(_host(ops.axpby(2.0, _dev(X), -3.0, _dev(Y))), 2.0 * X - 3.0 * Y)
        Xd = _dev(X)
        ops.hadamard_(Xd, _dev(Y))
        np.testing.assert_array_equal(_host(Xd), X * Y)
    for rows, cols in ((1, 1), (13, 300), (3, 5000), (200, 2)):
        X = _ints((rows, cols + 2), rng, dtype, -3, 4)
        got = float(_host(ops.norm1(_dev(X)[:, :cols]))[0])
        assert got == np.abs(X[:, :cols].astype(np.float64)).sum(0).max()
    u = U32 if dtype == np.float32 else U64
    for rows, cols in ((1, 7), (9, 1000), (4, 3000)):
        X = rng.uniform(-1, 1, (rows, cols)).astype(dtype)
        X[rows // 2] = 0
        Xd = _dev(X)
        ops.normalize_rows_(Xd)
        X64 = X.astype(np.float64)
        n = np.linalg.norm(X64, axis=1, keepdims=True)
        ref = np.where(n > 0, X64 / np.where(n > 0, n, 1), 0.0)
        err = np.abs(_host(Xd) - ref).max() / (4 * u)
        _record("normalize_rows_", err)
        assert err <= 1.0
        assert not _host(Xd)[rows // 2].any()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_row_sums_both_kernels(dtype):
    """row_sums on exact data: the warp-per-row kernel (cols < 2048), the CTA-per-row kernel (cols >= 2048, rows <= 65535) and
    the warp-per-row kernel again for rows > 65535 with wide columns; strided rows."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(9)
    for rows, cols in ((1, 1), (9, 2047), (3, 2048), (257, 5001), (65535, 2048), (65543, 2048)):
        Xh = rng.randint(0, 4, (rows, cols + 1), dtype=np.int8)
        X = _dev(Xh).to(torch.float32 if dtype == np.float32 else torch.float64)
        got = _host(ops.row_sums(X[:, :cols]))
        np.testing.assert_array_equal(got, Xh[:, :cols].sum(1, dtype=np.int64).astype(np.float64))


# =============================================================================================
# 4. element-wise MU terms, divergences and the Tucker core step
# =============================================================================================
BETAS = [0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.2]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("beta", BETAS)
def test_mu_terms(beta, dtype, sms):
    """P = K^(beta-2) X and Q = K^(beta-1) in all four kernel modes (beta = 1, 2, 3, general), at one block and past the grid-stride
    wrap, and P written over K with Q not wanted.  Bound: 16 units of the format relative (pow within a few ulp, one product)."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(int(beta * 10))
    u = U32 if dtype == np.float32 else U64
    for count in (1, 1001, 256 * sms * 16 * 2 + 5):
        K = (rng.rand(count) * 3 + 0.05).astype(dtype)
        X = (rng.rand(count) * 5).astype(dtype)
        X[::7] = 0
        K64, X64 = K.astype(np.float64), X.astype(np.float64)
        Pref, Qref = K64 ** (beta - 2) * X64, K64 ** (beta - 1)
        P, Q = ops.mu_terms(_dev(K), _dev(X), beta)
        for got, ref, tag in ((P, Pref, "P"), (Q, Qref, "Q")):
            err = (np.abs(_host(got) - ref) / (16 * u * np.abs(ref) + 1e-300)).max()
            _record(f"mu_terms {tag}", err)
            assert err <= 1.0, (tag, err)
        Kd = _dev(K)
        P2, Q2 = ops.mu_terms(Kd, _dev(X), beta, want_q=False, out_p=Kd)
        assert Q2 is None and P2.data_ptr() == Kd.data_ptr()
        np.testing.assert_array_equal(_host(Kd), _host(P))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_mu_apply(dtype):
    """max(F (num / den)^gamma, floor) with a matrix denominator and with a vector one per row and per column, on non-square shapes
    (swapping i / cols and i % cols changes the result); gamma != 1; the floor; NaN propagates.  Bound: 16 units of the format
    relative (a quotient, a pow, a product)."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(2)
    u = U32 if dtype == np.float32 else U64
    for rows, cols in ((3, 7), (64, 1001), (1001, 5)):
        F = rng.rand(rows, cols).astype(dtype)
        num = (rng.rand(rows, cols) * 2).astype(dtype)
        num[0, : cols // 2] = 0                                       # floor
        den_m = (rng.rand(rows, cols) + 0.1).astype(dtype)
        den_r = (rng.rand(rows) + 0.1).astype(dtype)
        den_c = (rng.rand(cols) + 0.1).astype(dtype)
        F64, n64 = F.astype(np.float64), num.astype(np.float64)
        for gamma in (1.0, 0.5, 1 / 3.2):
            for tag, d64 in (("mat", den_m.astype(np.float64)), ("row", den_r.astype(np.float64)[:, None]),
                             ("col", den_c.astype(np.float64)[None, :])):
                if tag == "mat":
                    got = ops.mu_apply(_dev(F), _dev(num), den_mat=_dev(den_m), gamma=gamma)
                else:
                    got = ops.mu_apply(_dev(F), _dev(num), den_vec=_dev(den_r if tag == "row" else den_c), vec_per_row=tag == "row",
                                       gamma=gamma)
                ref = np.maximum(F64 * (n64 / d64) ** gamma, 1e-12)
                g = _host(got)
                assert np.all(g[0, : cols // 2] == np.asarray(1e-12, dtype))
                err = (np.abs(g - ref) / (16 * u * ref)).max()
                _record("mu_apply", err)
                assert err <= 1.0, (rows, cols, gamma, tag, err)
        Fn = F.copy()
        Fn[rows // 2, cols // 2] = np.nan
        g = _host(ops.mu_apply(_dev(Fn), _dev(num), den_vec=_dev(den_c), floor=0.5))
        assert np.isnan(g[rows // 2, cols // 2]) and np.isnan(g).sum() == 1 and np.all(g[~np.isnan(g)] >= 0.5)


def _beta_components(a, b, beta):
    """Sum of the magnitudes of the parts each term of oracle.beta_divergence is formed from: the scale of its rounding error,
    which for a term near zero (a close to b) is far above the term itself."""
    with np.errstate(divide="ignore", invalid="ignore"):
        if beta == 1:
            return np.where(a != 0, np.abs(a * np.log(np.where(a != 0, a / b, 1.0))), 0.0) + a + b
        if beta == 0:
            return a / b + np.where(a != 0, np.abs(np.log(np.where(a != 0, a / b, 1.0))), 0.0) + 1.0
        return (a ** beta + abs(beta - 1.0) * b ** beta + beta * a * b ** (beta - 1.0)) / abs(beta * (beta - 1.0))


def _reduce_chain(count):
    """Longest chain of float64 additions behind one result of run_reduce (csrc/elementwise.cu): a thread's grid-stride terms, the
    256-thread tree of a block, one thread's share of the block partials and the tree again -- plus that of numpy's pairwise sum
    of the reference (blocks of at most 128 terms, then a binary tree)."""
    blocks = max(1, min(_cdiv(count, 256 * 4), 1184))
    kernel = _cdiv(count, blocks * 256) + 8 + _cdiv(blocks, 256) + 8
    return kernel + 128 + int(np.ceil(np.log2(count)))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("beta", [0.0, 0.5, 1.0, 1.5, 2.0, 3.0])
def test_beta_divergence_and_reductions(beta, dtype):
    """beta_divergence against oracle.beta_divergence on data with exact zeros in A, and sq_diff (with and without B) and dot
    against pairwise numpy sums, at one block, many blocks, and above RMAX_BLOCKS RB 4 elements (the grid-stride loop wraps).
    Both sides form the terms in float64 from the same stored values, so the bound is worst-case float64 arithmetic:
    2^-53 (8 + chain) S, with 8 units for a term (a log or pow of a few ulp and a few operations), `chain` the two summation
    orders of _reduce_chain, and S the sum of the magnitudes the terms are formed from."""
    from nn_fac import _ops as ops
    rng = np.random.RandomState(int(beta * 4))
    for count in (100, 300007, 1184 * 256 * 4 + 999):
        A = (rng.rand(count) * 4).astype(dtype)
        A[rng.rand(count) < 0.2] = 0
        B = (rng.rand(count) * 4 + 0.01).astype(dtype)
        S = (rng.rand(count) - 0.5).astype(dtype)
        A64, B64, S64 = A.astype(np.float64), B.astype(np.float64), S.astype(np.float64)
        k = (8 + _reduce_chain(count)) * U64
        cases = (("beta_divergence", ops.beta_divergence(_dev(A), _dev(B), beta), orc.beta_divergence(A64, B64, beta),
                  _beta_components(A64, B64, beta).sum()),
                 ("sq_diff", ops.sq_diff(_dev(A), _dev(B)), np.sum((A64 - B64) ** 2), np.sum((A64 - B64) ** 2)),
                 ("sq_diff without B", ops.sq_diff(_dev(A)), np.sum(A64 ** 2), np.sum(A64 ** 2)),
                 ("dot", ops.dot(_dev(A), _dev(S)), np.sum(A64 * S64), np.sum(np.abs(A64 * S64))))
        for name, got, ref, scale in cases:
            err = abs(float(_host(got)[0]) - float(ref)) / (k * float(scale))
            _record(name, err)
            assert err <= 1.0, (name, count, float(_host(got)[0]), float(ref))


def _pg_ref(core, MtX, Ms, step, sparse, delta, state, nsteps):
    """ntd.py:607-617 in float64: P = core x_0 M0 x_1 M1 x_2 M2, gradient -MtX + P + sparse, d = min(step g, core), core -= d,
    upd = ||d||; the loop `while cnt <= 300 and upd >= delta upd_0`, and a first step that moves nothing counts all 300.
    Returns the core and the state {upd_0, upd, cnt, done}."""
    core = core.astype(np.float64).copy()
    upd0, upd, cnt, done = state
    M64 = [M.astype(np.float64) for M in Ms]
    for _ in range(nsteps):
        if done:
            break
        P = orc.multi_mode_dot(core, M64)
        g = -MtX.astype(np.float64) + P + sparse
        d = np.minimum(step * g, core)
        core = core - d
        u = float(np.sqrt((d * d).sum()))
        if cnt == 1:
            upd0 = u
        upd = u
        cnt += 1
        done = not (cnt <= 300 and upd >= delta * upd0)
        if cnt == 2 and u == 0.0:
            cnt, done = 301, True
    return core, [upd0, upd, float(cnt), 1.0 if done else 0.0]


PG_RANKS = [(1, 1, 1), (64, 64, 64), (5, 64, 17), (64, 3, 64)]


def _pg_exact(ranks, dtype, rng):
    """Exact data for one step of size 1/4: integer core, non-symmetric integer M (a transposed M fails) and MtX = P + small
    integers, so that the step has both clamped and free entries and every value is an integer or quarter below 2^24."""
    core = rng.randint(0, 4, ranks).astype(np.float64)
    Ms = [rng.randint(0, 4, (r, r)).astype(np.float64) for r in ranks]
    P = orc.multi_mode_dot(core, Ms)
    assert np.abs(P).max() < 2 ** 24
    MtX = P + rng.randint(-8, 9, ranks)
    return core.astype(dtype), MtX.astype(dtype), [M.astype(dtype) for M in Ms]


def _pg_real(ranks, dtype, rng):
    """Data of a real Tucker core solve: M_n = A_n^T B_n (near a Gram, not symmetric), MtX from a sparse core, the step
    prod 1 / sigma_max(M_n) of ntd.py:590-594."""
    Ms = []
    for r in ranks:
        A = rng.rand(r + 6, r)
        Ms.append(A.T @ (A + 0.2 * rng.rand(r + 6, r)))
    truth = rng.rand(*ranks) * (rng.rand(*ranks) > 0.4)
    MtX = orc.multi_mode_dot(truth, Ms) + 0.1 * rng.randn(*ranks)
    step = 1.0
    for M in Ms:
        step /= np.linalg.svd(M, compute_uv=False)[0]
    core = rng.rand(*ranks)
    return core.astype(dtype), MtX.astype(dtype), [M.astype(dtype) for M in Ms], float(np.float32(step))


def _pg_launch(kind, c, MtX, Ms, Z, step, sparse, delta, state, dtype):
    from nn_fac import _ops as ops
    if kind == "step3":
        ops.core_pg_step3(c, MtX, Ms, Z, step, sparse, delta, state)
        return
    P = orc.multi_mode_dot(_host(c).astype(np.float64), [_host(M).astype(np.float64) for M in Ms]).astype(dtype)
    if kind == "dev":
        ops.core_pg_step_dev(c, MtX, _dev(P), delta, state)
    else:
        ops.core_pg_step(c, MtX, _dev(P), step, sparse, delta, state)


PG_KINDS = ["step3", "step", "dev"]
PG_REL = {np.float32: 2e-5, np.float64: 1e-12}


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("ranks", PG_RANKS)
@pytest.mark.parametrize("kind", PG_KINDS)
def test_core_pg_step_against_float64(kind, ranks, dtype):
    """core_pg_step3, and core_pg_step / core_pg_step_dev given P from numpy, against the float64 restatement of ntd.py:607-617,
    not against ops.multi_mode_dot:
      * one step on exact data must match bit for bit, core and state;
      * twelve steps of a real solve (non-symmetric M): relative Frobenius error of the core within 2e-5 in fp32 (1e-12 in
        fp64), cnt and done exact, upd_0 and upd within 10x that bound relative to |upd| + upd_0 (a converged core's last
        step is rounding noise)."""
    import torch
    rng = np.random.RandomState(sum(ranks))
    init = [0.0, 1.0, 1.0, 0.0]
    core, MtX, Ms = _pg_exact(ranks, dtype, rng)
    ref, st = _pg_ref(core, MtX, Ms, 0.25, 1.0, 1e-3, init, 1)
    c = _dev(core)
    state = torch.tensor(init + [0.25, 1.0], dtype=torch.float64, device="cuda")
    Md = [_dev(M) for M in Ms]
    _pg_launch(kind, c, _dev(MtX), Md, torch.empty_like(c), 0.25, 1.0, 1e-3, state, dtype)
    np.testing.assert_array_equal(_host(c), ref)
    np.testing.assert_allclose(_host(state)[:4], st, rtol=1e-15)

    core, MtX, Ms, step = _pg_real(ranks, dtype, rng)
    sparse = 0.01
    ref, st = _pg_ref(core, MtX, Ms, step, sparse, 1e-4, init, 12)
    c = _dev(core)
    state = torch.tensor(init + [step, sparse], dtype=torch.float64, device="cuda")
    Md, MtXd, Z = [_dev(M) for M in Ms], _dev(MtX), torch.empty_like(c)
    for _ in range(12):
        _pg_launch(kind, c, MtXd, Md, Z, step, sparse, 1e-4, state, dtype)
    rel = PG_REL[dtype]
    err = np.linalg.norm(_host(c) - ref) / np.linalg.norm(ref)
    _record(f"core_pg {np.dtype(dtype).name}", err / rel)
    assert err <= rel, err
    sh = _host(state)
    assert sh[2] == st[2] and sh[3] == st[3]
    # upd of a converged core is rounding noise: the bound is relative to the first step's size upd_0
    bound = rel * 10 * (np.abs(np.array(st[:2])) + st[0])
    _record(f"core_pg state {np.dtype(dtype).name}", (np.abs(sh[:2] - st[:2]) / bound).max())
    assert np.all(np.abs(sh[:2] - st[:2]) <= bound), (sh[:2], st[:2])


@pytest.mark.parametrize("kind", PG_KINDS)
@pytest.mark.parametrize("ranks", [(1, 1, 1), (5, 64, 17)])
def test_core_pg_stop_rules(ranks, kind):
    """A zero first step counts all 300 steps and stops (core_pg_finish_kernel); once `done` is set, a launch with a non-zero step
    changes neither the core nor the state; the delta rule stops the loop at the step where the float64 restatement stops, and
    the launches after it leave the core where the restatement's last step left it."""
    import torch
    rng = np.random.RandomState(4)
    core, MtX, Ms = _pg_exact(ranks, np.float64, rng)
    c = _dev(core)
    state = torch.tensor([0.0, 1.0, 1.0, 0.0, 0.0, 0.0], dtype=torch.float64, device="cuda")
    Md, Z = [_dev(M) for M in Ms], torch.empty_like(c)
    for _ in range(3):
        _pg_launch(kind, c, _dev(MtX), Md, Z, 0.0, 0.0, 0.1, state, np.float64)
    assert list(_host(state)[:4]) == [0.0, 0.0, 301.0, 1.0]
    assert _pg_ref(core, MtX, Ms, 0.0, 0.0, 0.1, [0.0, 1.0, 1.0, 0.0], 3)[1] == [0.0, 0.0, 301.0, 1.0]
    np.testing.assert_array_equal(_host(c), core)
    state[4] = 0.25                                   # a step that would move the core, were `done` not honoured
    _pg_launch(kind, c, _dev(MtX), Md, Z, 0.25, 0.0, 0.1, state, np.float64)
    np.testing.assert_array_equal(_host(c), core)
    assert list(_host(state)[:4]) == [0.0, 0.0, 301.0, 1.0]

    core, MtX, Ms, step = _pg_real(ranks, np.float64, rng)
    delta = 0.2
    ref, st = _pg_ref(core, MtX, Ms, step, 0.0, delta, [0.0, 1.0, 1.0, 0.0], 60)
    assert st[3] == 1.0 and 3 <= st[2] < 60, st
    c = _dev(core)
    state = torch.tensor([0.0, 1.0, 1.0, 0.0, step, 0.0], dtype=torch.float64, device="cuda")
    Md, Z = [_dev(M) for M in Ms], torch.empty_like(c)
    for _ in range(60):
        _pg_launch(kind, c, _dev(MtX), Md, Z, step, 0.0, delta, state, np.float64)
    sh = _host(state)
    assert sh[2] == st[2] and sh[3] == 1.0
    np.testing.assert_allclose(_host(c), ref, rtol=1e-12, atol=1e-13)
