"""The tensor-core HALS sweep (csrc/tc_sweep.cu, tc_sweep_kernel<RP, MT, LAG>) against float64.

This kernel runs every fp32 HALS solve at rank <= 128 whose columns fit in tensor memory: both solves of an NMF iteration, the
slice solves of the sharded path, the fp32 NTF / NTD / PARAFAC2 solves that fit.  Everything here calls nn_fac._ops on device
tensors (hals_nnls, hals_solve, hals_solve_slabs, NMFPlan.hals_solve); which instantiation ran is predicted by tc_plan (the launch
arithmetic of nnfac_tc_sweep_run restated from the device's SM count) and checked with torch.profiler, so a call that fell back
to the CUDA-core sweep fails.

Three kinds of check:
  * exact: the undo of the speculative blocks (a delta-stopped solve against the same solve with maxiter = its sweep count),
    column slices of a wide solve, power-of-two scaling, strided / aliased operands and installed operand planes must give the
    same bits;
  * element-wise rounding bounds evaluated in float64 along the oracle's own sweeps (_sweep_bound, derivation in its docstring);
  * stationarity of long solves against the CUDA-core fp32 solve of the same problem.
The worst error-to-bound ratio of every bounded test is printed at the end of the module (run with -s to see it).
"""
import contextlib
import re

import numpy as np
import pytest

from oracle import nnfac_oracle as orc

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
U16 = 2.0 ** -16
TILE = 128
_WORST = {}


def _record(name, ratio):
    _WORST[name] = max(_WORST.get(name, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    _close_router()
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


def _capture(fn):
    """Names of the CUDA kernels `fn` launched (torch.profiler, CUDA activity), or [] when the session delivered no device activity."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


# Profiling sessions of a long-lived process that has run many other tests can stop delivering device activity altogether.  The
# routing of nnfac_tc_sweep_run depends only on the entry point, r, n and the lag mode, so such a call is then profiled again in a
# fresh helper process (started on first need, ended with the module) on a synthetic problem of the same shape.
_ROUTER_SRC = r"""
import json, sys
sys.path[:0] = sys.argv[1:3]
import torch
from torch.profiler import ProfilerActivity, profile
from nn_fac import _lib as L, _ops as ops
lib, ctx = L.load_library(), L.ctx(torch.device("cuda", 0))
for line in sys.stdin:
    entry, r, n, mode = json.loads(line)
    b, V = torch.rand((r, n), device="cuda"), torch.rand((r, n), device="cuda")
    G, out = 2.0 * torch.eye(r, device="cuda"), torch.empty((r, n), device="cuda")
    res, scratch = torch.empty(4, dtype=torch.float64, device="cuda"), torch.empty(r * n, device="cuda")
    def run():
        if entry == "slabs":
            ops.hals_solve_slabs(b, n, 1, r * n, r, scratch, G, V, out, r, n, 1, 0.0, 0.0, res)
        else:
            ops.hals_solve(b, G, V, out, r, 1, 0.0, 0.0, res)
    L.check(lib.nnfac_ctx_sweep_variant(ctx, mode))
    names = []
    for _ in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        if names:
            break
    print(json.dumps(names), flush=True)
"""
_ROUTER = []


def _router_names(entry, r, n, mode):
    import json
    import os
    import subprocess
    import sys
    if not _ROUTER:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        _ROUTER.append(subprocess.Popen([sys.executable, "-c", _ROUTER_SRC, root, os.path.join(root, "nn-fac_b200")],
                                        stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True))
    proc = _ROUTER[0]
    proc.stdin.write(json.dumps([entry, int(r), int(n), int(mode)]) + "\n")
    proc.stdin.flush()
    line = proc.stdout.readline()
    assert line, "the routing helper process ended"
    return json.loads(line)


def _close_router():
    while _ROUTER:
        proc = _ROUTER.pop()
        proc.stdin.close()
        try:
            proc.wait(timeout=60)
        except Exception:
            proc.kill()
            proc.wait()


def _check_routing(fn, expect, entry, r, n, mode):
    """The tensor-core sweep `expect` = (RP, MT, LAG) and no CUDA-core sweep ran for `fn` (or, when this process's profiler
    records nothing, for the same entry point, shape and lag mode in the helper process)."""
    names = _capture(fn)
    if not names:
        names = _router_names(entry, r, n, mode)
    assert names, "the profiler recorded no CUDA activity, here and in a fresh process"
    assert _tc_kernels(names) == {expect}, (expect, sorted(set(names)))
    assert not any("hals_sweep" in nm or "gen_sweep" in nm for nm in names), sorted(set(names))


_TC_NAME = re.compile(r"tc_sweep_kernel<\s*(?:\(int\))?\s*(\d+)\s*,\s*(?:\(int\))?\s*(\d+)\s*,\s*(?:\(bool\))?\s*(\w+)\s*>")


def _tc_kernels(names):
    """The (RP, MT, LAG) instantiations of tc_sweep_kernel among the recorded kernel names."""
    out = set()
    for nm in names:
        m = _TC_NAME.search(nm)
        if m:
            out.add((int(m.group(1)), int(m.group(2)), m.group(3) in ("true", "1")))
    return out


# =============================================================================================
# launch arithmetic
# =============================================================================================
MAIL_COUNT = 1 << 18        # nnfac_ctx_create: mailbox words of a context
XMAXG = 160                 # board entries per rank (csrc/tc_sweep.cu)


def tc_plan(r, n, sms, lag_mode, collective=False):
    """nnfac_tc_sweep_run restated: None when the shape is outside the kernel, else padded rank, columns per CTA, grid, the
    instantiation (RP, MT, LAG), tiles of a full and of the last CTA, and the speculative blocks (NSPEC) of the variant."""
    if r > 128 or n < 1:
        return None
    rp = 64 if r <= 64 else 128
    max_cols = (256 // rp) * TILE
    cols = _cdiv(_cdiv(n, sms), 32) * 32
    if cols > max_cols:
        return None
    grid = _cdiv(n, cols)
    if 4 * grid * grid > MAIL_COUNT or grid > XMAXG:
        return None
    lag_possible = (collective or grid > 1) and (rp == 128 or cols <= 2 * TILE)
    lag_pays = collective or (cols <= TILE and grid >= 64)
    lag = lag_possible and (lag_mode >= 2 or (lag_mode == 1 and lag_pays))
    mt = 2 if (rp == 128 or lag or cols <= 2 * TILE) else 4
    last = n - (grid - 1) * cols
    nblk = _cdiv(r, 16)
    nspec = nblk if lag else min(nblk, 3 if rp == 64 else 6)
    return dict(rp=rp, cols=cols, grid=grid, kernel=(rp, mt, lag), mt=mt, lag=lag, tiles=_cdiv(cols, TILE), last_cols=last,
                last_tiles=_cdiv(last, TILE), nblk=nblk, nspec=nspec)


VARIANTS = {"64x2": (64, 2, False), "64x4": (64, 4, False), "64x2_lag": (64, 2, True), "128x2": (128, 2, False),
            "128x2_lag": (128, 2, True)}


def variant_layouts(name, sms):
    """Column counts (and the lag mode that selects the variant) for every CTA layout the instantiation allows: one tile per CTA
    with the second tile inactive, the most tiles per CTA, a ragged last CTA whose last tile is ragged, three of four tiles (MT = 4)
    and grid = 1 (plain variants; the lagged ones need a second CTA, grid = 2 instead)."""
    rp, mt, lag = VARIANTS[name]
    mode = 2 if lag else 0
    if mt == 4:
        ns = {"4 of 4 tiles": 512 * sms, "3 of 4 tiles": 384 * sms - 5, "ragged": 512 * sms - 77}
    else:
        ns = {"1 of 2 tiles": 100 * sms, "2 of 2 tiles": 256 * sms, "ragged": 256 * sms - 77,
              ("grid 2" if lag else "grid 1"): 40 if lag else 20}
    return mode, ns


def _check_layout(label, p, sms):
    if label.startswith("4 of 4"):
        assert p["tiles"] == 4 and p["last_cols"] == p["cols"], p
    elif label.startswith("3 of 4"):
        assert p["tiles"] == 3 and p["last_cols"] < p["cols"], p
    elif label.startswith("1 of 2"):
        assert p["tiles"] == 1 and p["grid"] > 1, p
    elif label.startswith("2 of 2"):
        assert p["tiles"] == 2 and p["last_cols"] == p["cols"], p
    elif label == "ragged":
        assert p["last_cols"] < p["cols"] and p["last_cols"] % TILE and p["last_tiles"] == p["tiles"], p
    elif label == "grid 1":
        assert p["grid"] == 1, p
    elif label == "grid 2":
        assert p["grid"] == 2, p


@contextlib.contextmanager
def sweep_variant(mode):
    """nnfac_ctx_sweep_variant: 0 plain stop test, 1 auto, 2 lagged wherever possible; the environment default again on exit."""
    import torch
    from nn_fac import _lib as L
    lib, ctx = L.load_library(), L.ctx(torch.device("cuda", torch.cuda.current_device()))
    L.check(lib.nnfac_ctx_sweep_variant(ctx, mode))
    try:
        yield
    finally:
        L.check(lib.nnfac_ctx_sweep_variant(ctx, -1))


def _solve(UtM, UtU, V0, r, maxiter, delta, sp=0.0, mode=0, expect=None):
    """hals_solve out of place on device copies under lag mode `mode`.  `expect`: the (RP, MT, LAG) that must have run (profiled)."""
    import torch
    from nn_fac import _ops as ops
    b, G, Vin = _dev(UtM), _dev(UtU), _dev(V0)
    V = torch.full_like(Vin, float("nan"))
    res = torch.full((4,), float("nan"), dtype=torch.float64, device="cuda")
    run = lambda: ops.hals_solve(b, G, Vin, V, r, maxiter, delta, sp, res)  # noqa: E731
    with sweep_variant(mode):
        if expect is not None:
            _check_routing(run, expect, "solve", r, UtM.shape[1], mode)
        else:
            run()
    return _host(V), _host(res)


# =============================================================================================
# problems and the float64 bound
# =============================================================================================
def _problem(r, n, seed, rho=0.5, kind="dominant"):
    """fp32 UtM, UtU, V0.  kind "dominant": a symmetric positive definite Gram with off-diagonal entries of both signs whose row
    sums of |G_kj| / G_kk stay below rho * 1.6 (diagonal scaling in [0.8, 1.25]), so that the rounding errors of one row reach the
    others damped and the element-wise bound stays tight; "nmf": U^T U of a non-negative U (all entries positive, as in an NMF).
    The right-hand side is G V* + noise with a sparse V*, so that the solution has active bounds and the steps are of the size
    of V."""
    rng = np.random.RandomState(seed)
    if kind == "dominant":
        E = rng.uniform(-1, 1, (r, r))
        E = (E + E.T) / 2
        np.fill_diagonal(E, 0)
        if r > 1:
            E *= rho / np.abs(E).sum(1).max()
        s = rng.uniform(0.8, 1.25, r) * np.sqrt(7.3)
        G = s[:, None] * (np.eye(r) + E) * s[None, :]
    else:
        U = rng.rand(2 * r + 8, r) + 0.05
        G = U.T @ U
    Vt = rng.rand(r, n) * (rng.rand(r, n) > 0.3)
    UtM = G @ Vt + 0.3 * np.sqrt(np.diag(G)).mean() * rng.randn(r, n)
    V0 = rng.rand(r, n)
    return UtM.astype(np.float32), G.astype(np.float32), V0.astype(np.float32)


def _sweep_bound(UtM, UtU, V0, sp=0.0, maxiter=1, delta=0.0, b_err=None, cols=None):
    """The float64 sweeps of nnls.py (oracle.hals_nnls_acc, restated so that it can carry a bound) on the columns `cols`, with an
    element-wise bound on |V_kernel - V|.  Returns (V, bound, eps, eps_bound, cnt, ambiguous).

    The kernel keeps the scaled residual W_k = (b_k - sp - G_k. V) / G_kk of every column in tensor memory and updates it; a row's
    new value is  V_k + max(W_k, -V_k) = max((b_k - sp - sum_{j != k} G_kj V_j) / G_kk, 0)  of the kernel's own V and W.  If the
    kernel's W differs from the exact residual of its V by a drift D_k, its new V_k differs from the float64 one by at most
        e_k = sum_{j != k} |G_kj| e_j / G_kk  +  D_k  +  I_k  +  2^-24 |V_k|          (propagation, drift, in-block, V + d)
    with e_j the current bounds of the other rows (already updated for j < k).  The drift accumulates over the call:
      * initial residual (UtM - sp) / G_kk plus the tensor-core product of the -G / diag planes with V, both split into three bf16
        terms (6 of 9 products, the dropped three below 2^-24 relative): r + 8 roundings (the r-term accumulation, b - sp, 1 / G_kk
        and the product, the plane entries G_kj * (-1 / G_jj)), each counted as a truncating fp32 rounding (2^-23):
        2 (r + 8) 2^-24 (|b_k| + sp + sum_j |G_kj| |V0_j|) / G_kk  (+ |b_err_k| / G_kk: error of a right-hand side summed in fp32);
      * every rank-16 update of a block (applied to every row): two bf16 terms of the step (|d - hi - mid| <= 2^-16 |d|) against two
        of the Gram, three products (the mid x mid one dropped, <= 2^-16): 3 2^-16 sum_{j in block} |G_kj| |d_j| / G_kk, plus one
        truncating rounding of the accumulator, 2 2^-24 T_k with T_k = (|b_k| + sp + sum_j |G_kj| |V_j|) / G_kk the size of W;
    and inside a block the rows see each other through 15 fp32 FMAs with coefficients -G_kj * (1 / G_kk) (two roundings):
        I_k = 18 2^-24 (T_k + sum_{j in block, j < k} |G_kj| |d_j| / G_kk).
    |d_j| is taken as |d_j| + e_j (old) + e_j (new).  Rows with G_kk = 0 are skipped (the kernel keeps Vin, error 0).
    eps (sum of squared steps of the last sweep over the columns `cols`): |eps_k - eps| <= sum (2 |d| + ed) ed with ed the bound of
    a step, plus the fp32 sums (an r-FMA chain, a warp tree, the CTA and grid sums: r + 181 roundings of at most eps).  The stop
    test of nnls.py:156 runs as in the oracle; `ambiguous` is set when a decision lies within those bounds of the threshold."""
    b, G = UtM.astype(np.float64), UtU.astype(np.float64)
    V = V0.astype(np.float64)
    if cols is not None:
        b, V = b[:, cols], V[:, cols]
    r, n = b.shape
    absG = np.abs(G)
    diag = np.diag(G).copy()
    inv = np.where(diag != 0, 1.0 / np.where(diag != 0, diag, 1.0), 0.0)
    absb = np.abs(b) + abs(sp)

    def size(Vabs):
        return (absb + absG @ Vabs) * inv[:, None]

    e = np.zeros_like(V)
    D = 2 * (r + 8) * U32 * size(np.abs(V))
    if b_err is not None:
        be = b_err if cols is None else b_err[:, cols]
        D += np.abs(be) * inv[:, None]
    eps0, eps, cnt, ambiguous, eps_b = 0.0, 1.0, 1, False, 0.0
    while eps >= delta * eps0 and cnt <= maxiter:
        nd, nd_err = 0.0, 0.0
        for B0 in range(0, r, 16):
            blk = list(range(B0, min(B0 + 16, r)))
            dab = np.zeros((len(blk), n))
            for i, k in enumerate(blk):
                if diag[k] == 0:
                    continue
                Tk = (absb[k] + absG[k] @ np.abs(V)) * inv[k]
                S2 = (absG[k, B0:k] @ dab[:i]) * inv[k] if i else 0.0
                prop = (absG[k] @ e - absG[k, k] * e[k]) * inv[k]
                d = np.maximum((b[k] - G[k] @ V - sp) * inv[k], -V[k])
                V[k] += d
                e_old = e[k].copy()
                e[k] = prop + D[k] + 18 * U32 * (Tk + S2) + U32 * np.abs(V[k])
                ed = e_old + e[k]
                dab[i] = np.abs(d) + ed
                nd += float(d @ d)
                nd_err += float(((2 * np.abs(d) + ed) * ed).sum())
            D += 3 * U16 * (absG[:, B0:B0 + len(blk)] @ dab) * inv[:, None] + 2 * U32 * size(np.abs(V))
        eb = nd_err + (r + 181) * U32 * (nd + nd_err)
        if cnt == 1:
            eps0, eps0_b = nd, eb
        eps, eps_b = nd, eb
        cnt += 1
        if delta > 0 and abs(eps - delta * eps0) <= eps_b + delta * eps0_b:
            ambiguous = True
        if nd == 0.0 and eps0 == 0.0:
            cnt = max(cnt, maxiter + 1)
            break
    return V, e, eps, eps_b, cnt, ambiguous


def _compare(name, V, res, UtM, UtU, V0, maxiter, delta, sp=0.0, b_err=None, cols=None):
    """Kernel V (and result, when all columns are compared) against _sweep_bound; records the worst ratio."""
    f = lambda x: x.astype(np.float64)  # noqa: E731
    assert res[2] == -1.0 and res[3] == res[1] - 1, res
    assert np.all(np.isfinite(V)) and np.all(V[np.diag(UtU) != 0] >= 0)
    if cols is None:
        Vo, bound, eps, eps_b, cnt, amb = _sweep_bound(UtM, UtU, V0, sp, maxiter, delta, b_err)
        Vr, eps_r, cnt_r, _ = orc.hals_nnls_acc(f(UtM), f(UtU), f(V0), maxiter=maxiter, delta=delta,
                                                sparsity_coefficient=sp or None)
        assert cnt == cnt_r and np.allclose(Vo, Vr, rtol=1e-9, atol=1e-9 * np.abs(Vr).max())
        if amb and int(res[1]) != cnt:
            # a stop decision within the rounding bound of the threshold may go either way: V is then a different sweep's
            assert abs(int(res[1]) - cnt) == 1, (name, res, cnt)
            _record(name + " count flips", 1e-300)
            return Vo, bound
        assert int(res[1]) == cnt, (name, res, cnt)
        if eps_b > 0 or eps > 0:
            re = abs(res[0] - eps) / max(eps_b, 1e-300)
            _record(name + " eps", re)
            assert re <= 1.0, (name, res[0], eps, eps_b)
        Vk = V
    else:
        Vo, bound, _, _, cnt, _ = _sweep_bound(UtM, UtU, V0, sp, maxiter, delta, b_err, cols)
        assert int(res[1]) == cnt, (name, res, cnt)
        Vk = V[:, cols]
    ratio = np.abs(Vk - Vo) / np.maximum(bound, 1e-300)
    _record(name + " V", ratio.max())
    assert ratio.max() <= 1.0, (name, np.unravel_index(ratio.argmax(), ratio.shape), ratio.max())
    return Vo, bound


def _cols(n, rng, k=1200):
    """A column subset for the float64 comparison of a wide solve: the first and last 130 columns and k random ones."""
    if n <= k + 260:
        return None
    return np.unique(np.concatenate([np.arange(130), np.arange(n - 130, n), rng.choice(n, k, replace=False)]))


# =============================================================================================
# every variant and CTA layout
# =============================================================================================
RANKS = {64: [1, 17, 48, 64], 128: [65, 100, 128]}


@pytest.mark.parametrize("variant,r", [(v, r) for v in VARIANTS for r in RANKS[VARIANTS[v][0]]])
def test_every_variant_and_layout(variant, r, sms):
    """Each of the five instantiations in each CTA layout it allows (variant_layouts): the kernel that ran is the predicted one,
    5 sweeps at delta = 0 are within the element-wise bound of _sweep_bound (kappa = 1) on a column subset, and a delta-stopped
    solve on the smallest layout matches the oracle's count and eps and is within the same bound."""
    mode, layouts = variant_layouts(variant, sms)
    rng = np.random.RandomState(r)
    for label, n in layouts.items():
        p = tc_plan(r, n, sms, mode)
        assert p is not None and p["kernel"] == VARIANTS[variant], (label, n, p)
        _check_layout(label, p, sms)
        UtM, UtU, V0 = _problem(r, n, r * 7 + n % 1009)
        V, res = _solve(UtM, UtU, V0, r, 5, 0.0, mode=mode, expect=p["kernel"])
        _compare(f"variant {variant} delta = 0", V, res, UtM, UtU, V0, 5, 0.0, cols=_cols(n, rng))
    n = min(layouts.values())
    UtM, UtU, V0 = _problem(r, n, r + 3)
    V, res = _solve(UtM, UtU, V0, r, 200, 0.01, mode=mode, expect=tc_plan(r, n, sms, mode)["kernel"])
    assert 3 <= res[1] < 200
    _compare(f"variant {variant} delta stop", V, res, UtM, UtU, V0, 200, 0.01)


# =============================================================================================
# one sweep, element by element
# =============================================================================================
ALL_RANKS = [1, 5, 16, 17, 33, 48, 63, 64, 65, 80, 100, 127, 128]


@pytest.mark.parametrize("sp", [0.0, 0.4])
@pytest.mark.parametrize("r", ALL_RANKS)
def test_single_sweep_elementwise(r, sp, sms):
    """maxiter = 1 element by element against the oracle's single sweep within _sweep_bound (kappa = 1).  The bound is about
    3 2^-16 of the steps of earlier blocks plus 2 (r + 8) 2^-24 of the initial residual's size: dropping one of the three products
    of a rank-16 update leaves an error of up to 2^-8 of a step term, far outside it.  Its size relative to V is recorded as
    "single sweep bound / 5e-4" (the norm-wise tolerance of the older whole-solve tests)."""
    n = 3001
    UtM, UtU, V0 = _problem(r, n, 31 * r + int(sp * 10))
    V, res = _solve(UtM, UtU, V0, r, 1, 0.01, sp=sp, mode=0, expect=tc_plan(r, n, sms, 0)["kernel"])
    assert res[1] == 2
    Vo, bound = _compare("single sweep elementwise", V, res, UtM, UtU, V0, 1, 0.01, sp=sp)
    _record("single sweep bound / 5e-4", np.linalg.norm(bound) / np.linalg.norm(Vo) / 5e-4)


# =============================================================================================
# undo of the speculative blocks
# =============================================================================================
UNDO = [("64x2", 5), ("64x2", 17), ("64x2", 48), ("64x2", 64), ("64x4", 33), ("64x4", 64), ("64x2_lag", 17), ("64x2_lag", 64),
        ("128x2", 65), ("128x2", 96), ("128x2", 128), ("128x2_lag", 80), ("128x2_lag", 128)]


@pytest.mark.parametrize("variant,r", UNDO)
def test_undo_of_speculative_blocks_is_exact(variant, r, sms):
    """A delta-stopped solve that returns count c ran the first NSPEC blocks of sweep c (all of them with the lagged stop test, or
    when nblk <= NSPEC) and undid them: it must equal, bit for bit in V and in all four result entries, the solve with
    maxiter = c - 1, which speculates nothing at its end.  Masters parked in the idle operand plane (blocks 0, 1), in bk_extra
    (blocks 2, 3 of the lagged RP = 128 variant) and in registers (the rest) are all restored here.  Lag modes 0 and 2."""
    mode, layouts = variant_layouts(variant, sms)
    for label, n in layouts.items():
        p = tc_plan(r, n, sms, mode)
        if p["grid"] < 2:
            continue
        assert p["kernel"] == VARIANTS[variant]
        UtM, UtU, V0 = _problem(r, n, r * 5 + n % 313, kind="nmf")
        Va, ra = _solve(UtM, UtU, V0, r, 300, 0.01, mode=mode, expect=p["kernel"])
        c = int(ra[1])
        assert 3 <= c < 300, ra
        Vb, rb = _solve(UtM, UtU, V0, r, c - 1, 0.01, mode=mode)
        np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(Va, Vb)


# =============================================================================================
# column-slice invariance
# =============================================================================================
@pytest.mark.parametrize("r,n,slices", [(48, 40000, [(12345, 1000, 0), (3001, 8192, 2), (39970, 20, 0), (7, 1000, 2)]),
                                        (100, 30000, [(12345, 1000, 0), (3001, 8192, 2), (29980, 20, 0), (777, 130, 2)])])
def test_column_slices_equal_the_wide_solve(r, n, slices, sms):
    """At delta = 0 and fixed maxiter every column is solved on its own: V[:, a:a+w] of a wide solve equals bit for bit the solve
    of those columns alone, on another variant, grid and tile position (four-tile n = 40000 at r = 48; slices of 1000, 8192
    (lagged), 20 (grid 1) columns).  Expected exact: every accumulator row of an MMA is its own column."""
    UtM, UtU, V0 = _problem(r, n, r + n)
    pw = tc_plan(r, n, sms, 0)
    V, _ = _solve(UtM, UtU, V0, r, 6, 0.0, mode=0, expect=pw["kernel"])
    seen = {pw["kernel"]}
    for a, w, mode in slices:
        p = tc_plan(r, w, sms, mode)
        Vs, _ = _solve(UtM[:, a:a + w], UtU, V0[:, a:a + w], r, 6, 0.0, mode=mode, expect=p["kernel"])
        seen.add(p["kernel"])
        np.testing.assert_array_equal(Vs, V[:, a:a + w], err_msg=f"slice {a}:{a + w}")
    assert len(seen) >= 2, seen


# =============================================================================================
# power-of-two scaling
# =============================================================================================
@pytest.mark.parametrize("r,n,mode", [(17, 5000, 0), (64, 20000, 2), (48, 40000, 0), (100, 9000, 0), (128, 12000, 2)])
def test_power_of_two_scaling(r, n, mode, sms):
    """Every operation of the sweep is homogeneous: with UtM, UtU (and sp) scaled by 2^+-30, V, count and eps must keep their bits;
    with UtM, V0 (and sp) scaled by 2^k, V must scale exactly and eps by 2^2k.  An absolute constant anywhere fails."""
    UtM, UtU, V0 = _problem(r, n, r * 3 + n, kind="nmf")
    sp = 0.25
    V, res = _solve(UtM, UtU, V0, r, 40, 0.01, sp=sp, mode=mode, expect=tc_plan(r, n, sms, mode)["kernel"])
    for s in (2.0 ** 30, 2.0 ** -30):
        Vs, rs = _solve(UtM * np.float32(s), UtU * np.float32(s), V0, r, 40, 0.01, sp=sp * s, mode=mode)
        np.testing.assert_array_equal(Vs, V)
        np.testing.assert_array_equal(rs, res)
    for k in (20, -20):
        s = np.float32(2.0 ** k)
        Vs, rs = _solve(UtM * s, UtU, V0 * s, r, 40, 0.01, sp=sp * 2.0 ** k, mode=mode)
        np.testing.assert_array_equal(Vs, V * s)
        assert rs[0] == res[0] * 2.0 ** (2 * k) and list(rs[1:]) == list(res[1:])


# =============================================================================================
# sparsity, zero diagonals, negative starts
# =============================================================================================
@pytest.mark.parametrize("sp", [0.05, 0.4])
@pytest.mark.parametrize("r,n,mode", [(50, 3001, 0), (50, 20000, 2), (100, 9000, 0), (127, 9000, 2)])
def test_sparsity_zero_diagonals_negative_starts(r, n, mode, sp, sms):
    """Sparsity (b - sp) * invd, rows with a zero diagonal (zero row and column of UtU, as from a zero column of U) in the first
    block, a middle block and the last, partial block, with negative start values on those rows.  5 sweeps at delta = 0 and a
    delta-stopped solve within _sweep_bound; the skipped rows keep Vin bit for bit, out of place and in place."""
    import torch
    from nn_fac import _ops as ops
    UtM, UtU, V0 = _problem(r, n, r + n + int(sp * 100))
    skip = [3, 16 * (r // 32) + 5, r - 1]
    for k in skip:
        UtU[k, :] = 0
        UtU[:, k] = 0
        V0[k, ::2] *= -1
    kern = tc_plan(r, n, sms, mode)["kernel"]
    rng = np.random.RandomState(r)
    for maxiter, delta in ((5, 0.0), (200, 0.01)):
        V, res = _solve(UtM, UtU, V0, r, maxiter, delta, sp=sp, mode=mode, expect=kern)
        np.testing.assert_array_equal(V[skip], V0[skip])
        _compare(f"sparsity {sp} zero diag", V, res, UtM, UtU, V0, maxiter, delta, sp=sp,
                 cols=_cols(n, rng) if delta == 0 else None)
        Vi = _dev(V0)
        with sweep_variant(mode):
            ri = ops.hals_solve(_dev(UtM), _dev(UtU), Vi, Vi, r, maxiter, delta, sp,
                                torch.empty(4, dtype=torch.float64, device="cuda"))
        np.testing.assert_array_equal(_host(Vi), V)
        np.testing.assert_array_equal(_host(ri), res)


# =============================================================================================
# operand addressing
# =============================================================================================
@pytest.mark.parametrize("r,n,mode", [(5, 1001, 0), (64, 20000, 2), (33, 40000, 0), (100, 9000, 2), (128, 37, 0)])
def test_strided_operands_and_aliasing(r, n, mode, sms):
    """UtM and Vin as column slices of NaN-filled buffers (ld > n, an offset that is not 16-byte aligned), V written into one with
    ld > n, UtU a sub-block of a NaN-filled r + 3 x r + 5 buffer: the result equals the contiguous solve bit for bit, no NaN is
    read and no padding is written.  In place (Vin aliasing V) equals out of place.  The contiguous solve is within _sweep_bound."""
    import torch
    from nn_fac import _ops as ops
    UtM, UtU, V0 = _problem(r, n, 3 * r + n)
    kern = tc_plan(r, n, sms, mode)["kernel"]
    Vc, rc = _solve(UtM, UtU, V0, r, 6, 0.0, sp=0.1, mode=mode, expect=kern)
    _compare("strided contiguous", Vc, rc, UtM, UtU, V0, 6, 0.0, sp=0.1, cols=_cols(n, np.random.RandomState(r)))
    nan = float("nan")
    off = 3
    ld = n + 11
    bb = torch.full((r, ld), nan, device="cuda")
    vb = torch.full((r, ld), nan, device="cuda")
    ob = torch.full((r + 2, ld + 6), nan, device="cuda")
    gb = torch.full((r + 3, r + 5), nan, device="cuda")
    bb[:, off:off + n] = _dev(UtM)
    vb[:, off:off + n] = _dev(V0)
    gb[1:r + 1, 2:r + 2] = _dev(UtU)
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    with sweep_variant(mode):
        _check_routing(lambda: ops.hals_solve(bb[:, off:off + n], gb[1:r + 1, 2:r + 2], vb[:, off:off + n], ob[1:r + 1, 5:5 + n], r,
                                              6, 0.0, 0.1, res), kern, "solve", r, n, mode)
    oh = _host(ob)
    np.testing.assert_array_equal(oh[1:r + 1, 5:5 + n], Vc)
    np.testing.assert_array_equal(_host(res), rc)
    mask = np.ones(oh.shape, bool)
    mask[1:r + 1, 5:5 + n] = False
    assert np.isnan(oh[mask]).all()
    vh, bh, gh = _host(vb), _host(bb), _host(gb)
    np.testing.assert_array_equal(vh[:, off:off + n], V0)
    np.testing.assert_array_equal(bh[:, off:off + n], UtM)
    assert np.isnan(vh[:, :off]).all() and np.isnan(vh[:, off + n:]).all() and np.isnan(bh[:, off + n:]).all()
    with sweep_variant(mode):
        ops.hals_solve(bb[:, off:off + n], gb[1:r + 1, 2:r + 2], vb[:, off:off + n], vb[:, off:off + n], r, 6, 0.0, 0.1, res)
    vh = _host(vb)
    np.testing.assert_array_equal(vh[:, off:off + n], Vc)
    np.testing.assert_array_equal(_host(res), rc)
    assert np.isnan(vh[:, :off]).all() and np.isnan(vh[:, off + n:]).all()


# =============================================================================================
# split right-hand side
# =============================================================================================
@pytest.mark.parametrize("nslabs", [1, 3, 7])
@pytest.mark.parametrize("r,n,mode", [(17, 3001, 0), (64, 20000, 2), (100, 9000, 0)])
def test_split_rhs_against_float64(r, n, mode, nslabs, sms):
    """hals_solve_slabs: the right-hand side is the sum of nslabs slabs [r_pad x ld], added in slab order in fp32 by the solve;
    rows r .. r_pad of every slab hold NaN, which must never be read.  Compared with the float64 solve of the float64 slab sum;
    the fp32 sum adds at most (nslabs - 1) 2^-24 sum |slab| to b (b_err of _sweep_bound)."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(r + nslabs)
    UtM, UtU, V0 = _problem(r, n, r * nslabs + n)
    r_pad = _cdiv(r, 16) * 16 + 16
    ld = n + 5
    parts = (rng.rand(nslabs, r, n) + 0.5).astype(np.float32)
    parts *= (UtM / parts.sum(0)).astype(np.float32)[None]
    slabs = np.full((nslabs, r_pad, ld), np.nan, np.float32)
    slabs[:, :r, :n] = parts
    total = parts.astype(np.float64).sum(0)
    b_err = (nslabs - 1) * U32 * np.abs(parts.astype(np.float64)).sum(0)
    kern = tc_plan(r, n, sms, mode)["kernel"]
    V = torch.empty((r, n), device="cuda")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    sd, Gd, Vin = _dev(slabs), _dev(UtU), _dev(V0)
    for maxiter, delta in ((5, 0.0), (200, 0.01)):
        with sweep_variant(mode):
            _check_routing(lambda: ops.hals_solve_slabs(sd, ld, nslabs, r_pad * ld, r_pad, torch.empty(r * n, device="cuda"), Gd, Vin,
                                                        V, r, n, maxiter, delta, 0.0, res), kern, "slabs", r, n, mode)
        _compare(f"split rhs {nslabs} slabs", _host(V), _host(res), total, UtU, V0, maxiter, delta, b_err=b_err,
                 cols=_cols(n, rng) if delta == 0 else None)
    np.testing.assert_array_equal(_host(Vin), V0)


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("r", [17, 64, 100])
def test_plan_solve_from_split_partials_against_float64(r, which, sms):
    """NMFPlan.hals_solve(which, None, ...) after fused(which, 0, keep_partials=True) adds the split-K partials in the order of the
    reduction kernel, i.e. solves for exactly plan.reduce(which): within _sweep_bound of the float64 solve of that right-hand side."""
    import torch
    from nn_fac import _ops as ops
    rng = np.random.RandomState(r + which)
    m, n = 3001, 1777
    X = torch.from_numpy((rng.rand(m, r) @ rng.rand(r, n) + 0.3 * rng.rand(m, n)).astype(np.float32)).cuda()
    Ut = torch.from_numpy(rng.rand(r, m).astype(np.float32)).cuda()
    V = torch.from_numpy(rng.rand(r, n).astype(np.float32)).cuda()
    plan = ops.NMFPlan(X).bind_rank(r)
    plan.set_factor(0, Ut)
    plan.set_factor(1, V)
    F = Ut if which == 0 else V
    G = ops.gram(V if which == 0 else Ut)
    plan.fused(which, 0, keep_partials=True)
    rhs = _host(plan.reduce(which))
    plan.fused(which, 0, keep_partials=True)
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    out = plan.hals_solve(which, None, G, F, 6, 0.0, 0.0, res)
    assert out is not None
    _compare("plan solve from partials", _host(out), _host(res), rhs, _host(G), _host(F), 6, 0.0)


# =============================================================================================
# operand planes installed by the solve
# =============================================================================================
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("r", [17, 64, 100])
def test_installed_planes_equal_set_factor(r, which, mode, monkeypatch):
    """plan.hals_solve(which, ...) writes the bf16 planes of its result itself (K-major hi / lo, and the row planes the fused passes
    read); skipped rows get their start value, undone speculative blocks their restored masters.  After a stale factor is
    installed, solve-and-install must leave the plan in the state of set_factor(which, result): every pass that reads factor
    `which` -- cross(1 - which, None), fused(1 - which, 0), fused(which, 0), fused(which, 1) at r <= 64 -- gives the same bits.
    m, n not multiples of 128, sparsity, a zero-diagonal row, a delta-stopped solve."""
    import torch
    from nn_fac import _ops as ops
    monkeypatch.setenv("NNFAC_MU_F32", "0")
    rng = np.random.RandomState(r * 3 + which)
    m, n = 1000, 2777
    U = rng.rand(m, r).astype(np.float32) + 0.05
    Vt = rng.rand(r, n).astype(np.float32) + 0.05
    X = torch.from_numpy(((U @ Vt) * (1 + 0.2 * rng.rand(m, n)) + 1e-3).astype(np.float32)).cuda()
    Ut = _dev(np.ascontiguousarray(U.T))
    Vd = _dev(Vt)
    len_w = m if which == 0 else n
    other = Vd if which == 0 else Ut
    stale = _dev(rng.rand(r, len_w).astype(np.float32) * 3)
    F0 = _dev(rng.rand(r, len_w).astype(np.float32))
    G = _host(ops.gram(other))
    G[r // 2, :] = 0
    G[:, r // 2] = 0
    Gd = _dev(G)
    rhs = ops.matmul(other, X.T.contiguous()) if which == 0 else ops.matmul(other, X)
    plans = [ops.NMFPlan(X).bind_rank(r) for _ in range(2)]
    for p in plans:
        p.set_factor(1 - which, other)
        p.set_factor(which, stale)
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    with sweep_variant(mode):
        out = plans[0].hals_solve(which, rhs, Gd, F0, 200, 0.01, 0.05, res)
    assert out is not None
    assert 3 <= res[1].item() < 200
    np.testing.assert_array_equal(_host(out)[r // 2], _host(F0)[r // 2])
    plans[1].set_factor(which, out)
    outs = []
    for p in plans:
        o = [p.cross(1 - which, None).clone()]
        for side, fm in ((1 - which, 0), (which, 0)) + (((which, 1),) if r <= 64 else ()):
            a, c = p.fused(side, fm)
            o += [a.clone(), c.clone()]
        outs.append(o)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# =============================================================================================
# long solves
# =============================================================================================
def _stationarity(V, b, G, sp):
    """||min(V, G V - b + sp)|| / ||b|| in float64 (zero at a solution of the NNLS problem)."""
    V, b, G = (x.astype(np.float64) for x in (V, b, G))
    return np.linalg.norm(np.minimum(V, G @ V - b + sp)) / np.linalg.norm(b)


@pytest.mark.parametrize("kind", ["dominant", "cond1e4"])
@pytest.mark.parametrize("r", [64, 128])
def test_long_solves(r, kind, sms):
    """500 sweeps at delta = 0: the residual is never re-formed, so its drift over the call is what limits the result.  By the
    derivation of _sweep_bound the drift of row k is at most 3 2^-16 sum_j |G_kj| sum_s |d_j^(s)| / G_kk (every rank update) plus
    2 (r + 8 + 500 nblk) 2^-24 T_k (one truncating rounding per update), and a step adds the in-block and V + d roundings,
    19 2^-24 T_k; at a fixed point of the kernel's sweep |min(V, G V - b)|_k <= G_kk * drift_k.  So the
    stationarity of the tensor-core solve must stay within 2 x that of the CUDA-core fp32 solve (which re-forms the residual) plus
    ||G_kk drift|| / ||b||, with sum_s |d^(s)| taken along the CUDA-core solve's 500 sweeps.  Well-conditioned problem: V within
    (||G_kk drift|| + stationarity gaps) / lambda_min(G) of the float64 solve (strong convexity)."""
    import torch
    from nn_fac import _ops as ops
    n = 2048
    rng = np.random.RandomState(r)
    if kind == "dominant":
        UtM, UtU, V0 = _problem(r, n, r + 1)
    else:
        base = rng.rand(3 * r, 1)
        Uc = base + (0.4 if r == 64 else 0.6) * rng.rand(3 * r, r)       # correlated columns of U
        G = Uc.T @ Uc
        c = np.linalg.cond(G)
        Vt = rng.rand(r, n) * (rng.rand(r, n) > 0.3)
        UtM = (G @ Vt + 0.05 * np.sqrt(np.diag(G)).mean() * rng.randn(r, n)).astype(np.float32)
        UtU, V0 = G.astype(np.float32), rng.rand(r, n).astype(np.float32)
        assert 3e3 < c < 3e4, c
    Vt_, rt = _solve(UtM, UtU, V0, r, 500, 0.0, mode=1, expect=tc_plan(r, n, sms, 1)["kernel"])
    assert rt[1] == 501
    # CUDA-core fp32 solve, one sweep per call, to collect sum_s |d^(s)| (on the device)
    Vc = _dev(V0)
    prev = Vc.clone().double()
    steps = torch.zeros_like(prev)
    bd, Gd = _dev(UtM), _dev(UtU)
    for _ in range(500):
        ops.hals_nnls(bd, Gd, Vc, r, 1, 0.0, 0.0, False, False, no_tc=True)
        cur = Vc.double()
        steps += (cur - prev).abs()
        prev = cur
    steps, prev = _host(steps), _host(prev)
    G64 = UtU.astype(np.float64)
    diag = np.diag(G64)
    T = (np.abs(UtM) + np.abs(G64) @ np.abs(prev)) / diag[:, None]
    nblk = _cdiv(r, 16)
    drift = 3 * U16 * (np.abs(G64) @ steps) / diag[:, None] + (2 * (r + 8 + 500 * nblk) + 19) * U32 * T
    gap = np.linalg.norm(diag[:, None] * drift) / np.linalg.norm(UtM.astype(np.float64))
    s_tc, s_cc = _stationarity(Vt_, UtM, UtU, 0.0), _stationarity(prev, UtM, UtU, 0.0)
    ratio = s_tc / (2 * s_cc + gap)
    _record(f"long solve stationarity {kind}", ratio)
    assert ratio <= 1.0, (s_tc, s_cc, gap)
    if kind == "dominant":
        Vo, _, _, _ = orc.hals_nnls_acc(UtM.astype(np.float64), G64, V0.astype(np.float64), maxiter=500, delta=0.0)
        lam = np.linalg.eigvalsh(G64).min()
        nb = np.linalg.norm(UtM.astype(np.float64))
        bound = (np.linalg.norm(diag[:, None] * drift) + (s_tc + _stationarity(Vo, UtM, UtU, 0.0)) * nb) / lam
        ev = np.linalg.norm(Vt_ - Vo) / bound
        _record("long solve V", ev)
        assert ev <= 1.0, (np.linalg.norm(Vt_ - Vo), bound)


# =============================================================================================
# stop rule edges
# =============================================================================================
@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("r,n", [(5, 3001), (64, 20000), (100, 9000)])
def test_stop_rule_edges(r, n, mode, sms):
    """UtM = 0 from V0 = 0: the first sweep moves nothing and the count is maxiter + 1 as in the oracle (eps = 0); maxiter in
    {1, 2, 3} x delta in {0, 0.5}: the oracle's count, eps and V (within _sweep_bound); result[2] = -1, result[3] = result[1] - 1."""
    kern = tc_plan(r, n, sms, mode)["kernel"]
    Z = np.zeros((r, n), np.float32)
    UtM, UtU, V0 = _problem(r, n, r + n)
    for maxiter in (1, 4, 9):
        V, res = _solve(Z, UtU, Z, r, maxiter, 0.01, mode=mode, expect=kern if maxiter == 1 else None)
        assert not V.any() and list(res) == [0.0, maxiter + 1.0, -1.0, float(maxiter)], res
    rng = np.random.RandomState(n)
    for maxiter in (1, 2, 3):
        for delta in (0.0, 0.5):
            V, res = _solve(UtM, UtU, V0, r, maxiter, delta, mode=mode)
            _compare("stop rule edges", V, res, UtM, UtU, V0, maxiter, delta, cols=_cols(n, rng) if delta == 0 else None)


# =============================================================================================
# generation wrap of the mailbox tags
# =============================================================================================
def test_generation_wrap_clears_the_mailboxes(sms):
    """The 16-bit call generation in the mailbox tags wraps after 65 535 solves, and sweep_prep_kernel clears the mailboxes then.
    Solve A1 (many CTAs), then exactly 65 534 single-CTA solves (n <= 32: they advance the generation but post nothing), then A2
    with other data on the same grid: A2 runs under A1's generation, after the clear, and must equal A2 solved on its own."""
    import torch
    from nn_fac import _ops as ops
    r, n = 64, 20000
    p = tc_plan(r, n, sms, 0)
    assert p["grid"] >= 2 and tc_plan(r, 20, sms, 0)["grid"] == 1
    A1 = _problem(r, n, 1, kind="nmf")
    A2 = _problem(r, n, 2, kind="nmf")
    ref, rref = _solve(*A2, r, 200, 0.01, mode=0, expect=p["kernel"])
    fb, fG, fV = _dev(A1[0][:, :20]), _dev(A1[1]), _dev(A1[2][:, :20])
    fo = torch.empty_like(fV)
    fres = torch.empty(4, dtype=torch.float64, device="cuda")
    _solve(*A1, r, 200, 0.01, mode=0)
    with sweep_variant(0):
        for _ in range(65534):
            ops.hals_solve(fb, fG, fV, fo, r, 1, 0.0, 0.0, fres)
    V2, r2 = _solve(*A2, r, 200, 0.01, mode=0)
    np.testing.assert_array_equal(r2, rref)
    np.testing.assert_array_equal(V2, ref)
