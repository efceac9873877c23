"""Accelerated HALS NNLS on the GPU (reference: nn_fac/update_rules/nnls.py:24-198).

The sweep loop runs in one persistent cooperative kernel (csrc/hals_sweep.cuh).  The reference's
wall-clock rule (``cnt <= 1 + alpha*rho`` with ``rho = atime/btime``, nnls.py:156,187-194) is
meaningless on a GPU and irreproducible on a CPU, so ``atime`` and ``alpha`` are accepted and
ignored: the deterministic rule (alpha = inf) always applies and ``rho`` is returned as 1e5.
"""
import numpy as np
import torch

import nn_fac.utils.errors as err
from nn_fac import _lib as L
from nn_fac import _ops as ops

_RHO_UNUSED = 100000  # nnls.py:149


def hals_nnls_device(UtM, UtU, V, r=None, maxiter=500, delta=0.01, sparsity_coefficient=None,
                     normalize=False, nonzero=False, result=None):
    """In-place solve on device tensors (UtM r x n, UtU r x r, V r x n).  Returns the device
    result vector {eps, cnt, zero_diag_row, sweeps}; nothing is synchronised."""
    r = UtM.shape[0] if r is None else r
    sp = 0.0 if sparsity_coefficient is None else float(sparsity_coefficient)
    return ops.hals_nnls(UtM, UtU, V, r, int(maxiter), delta, sp, bool(normalize), bool(nonzero), result)


def raise_if_zero_column(result_host):
    if result_host[2] >= 0:
        raise err.ZeroColumnWhenUnautorized(
            "Column " + str(int(result_host[2])) + " of U is zero with nonzero condition")


def hals_nnls_acc(UtM, UtU, in_V, maxiter=500, atime=None, alpha=0.5, delta=0.01,
                  sparsity_coefficient=None, normalize=False, nonzero=False):
    """Drop-in for nnls.hals_nnls_acc: returns (V, eps, cnt, rho) with V a fresh array.

    UtM: r x n, UtU: at least r x r, in_V: at least r x n (only the first r rows are used,
    tests/nnls_tests.py:40-47).  An empty in_V triggers the least-squares start of nnls.py:138-145.
    """
    V, eps, cnt, rho = _hals_nnls_acc(UtM, UtU, in_V, maxiter, delta, sparsity_coefficient, normalize, nonzero)
    return L.as_output(V), eps, cnt, rho


def _hals_nnls_acc(UtM, UtU, in_V, maxiter=500, delta=0.01, sparsity_coefficient=None, normalize=False, nonzero=False):
    """hals_nnls_acc with V in the working dtype (callers that keep computing with it: parafac2)."""
    for name, arg in (("UtM", UtM), ("UtU", UtU), ("in_V", in_V)):
        if len(np.shape(arg)) != 2:                                        # nnls.py:130-135
            raise err.ArgumentException(
                f"Argument {name} is an array of {np.shape(arg)} dimensions when it should be a matrix.")
    dt = L.resolve_dtype(UtM, UtU, in_V)
    b = L.to_device(UtM, dt)
    G = L.to_device(UtU, dt)
    r, n = b.shape
    if not np.prod(np.shape(in_V)):                                        # nnls.py:138-145
        V = torch.linalg.solve(G[:r, :r].double(), b.double())
        V.clamp_(min=0)
        scale = (b.double() * V).sum() / (G[:r, :r].double() * (V @ V.T)).sum()
        V = (V * scale).to(dt).contiguous()
    else:
        V = L.to_device(in_V, dt)                                          # the copy of nnls.py:147
        if V.data_ptr() == (in_V.data_ptr() if isinstance(in_V, torch.Tensor) else 0):
            V = V.clone()
    if G.shape[1] > r and V.shape[0] == G.shape[1]:
        # nnls.py:163/167 multiply the WHOLE row UtU[k,:] with V: rows >= r of in_V are never updated but enter every product
        # (tests/nnls_tests.py:44-45).  They are constants of the solve: fold them into the right-hand side.
        b = ops.axpby(1.0, b, -1.0, ops.matmul(G[:r, r:].contiguous(), V[r:, :].contiguous()))
    res = hals_nnls_device(b, G, V, r, maxiter, delta, sparsity_coefficient, normalize, nonzero).cpu().numpy()
    raise_if_zero_column(res)
    out = V if isinstance(in_V, torch.Tensor) else V.cpu().numpy()
    return out, np.float64(res[0]), int(res[1]), _RHO_UNUSED


def hals_coupling_nnls_acc(UtM, UtU, in_V, Vtarget, mu, maxiter=500, atime=None, alpha=0.5, delta=0.01,
                           normalize=False, nonzero=False):
    """Drop-in for nnls.hals_coupling_nnls_acc (nnls.py:204-352): min_{V >= 0} ||M - U V||^2 + mu ||V - Vtarget||^2, the
    flexible-coupling solve of nonnegative PARAFAC2 (parafac2.py:522).  Returns (V, eps, cnt, rho).

    The update of row k (nnls.py:318) is
        max((UtM[k] - UtU[k,:] V + mu (Vtarget[k] - V[k])) / (UtU[k,k] + mu), -V[k])
      = max(((UtM + mu Vtarget)[k] - (UtU + mu I)[k,:] V) / (UtU + mu I)[k,k], -V[k]),
    i.e. the plain sweep of hals_nnls_acc on the right-hand side UtM + mu Vtarget and the Gram UtU + mu I -- same kernels,
    same stop rule.  Rows whose UtU[k,k] is zero are skipped by the reference (nnls.py:316) although UtU[k,k] + mu is not:
    their diagonal entry is left at zero here, which is what makes the sweep skip them.  As for hals_nnls_acc, the
    deterministic stop rule always applies (`atime` / `alpha` are accepted and ignored); the reference raises ValueError
    (not ZeroColumnWhenUnautorized) for a zero column under `nonzero` (nnls.py:330)."""
    V, eps, cnt, rho = _hals_coupling_nnls_acc(UtM, UtU, in_V, Vtarget, mu, maxiter, delta, normalize, nonzero)
    return L.as_output(V), eps, cnt, rho


def _hals_coupling_nnls_acc(UtM, UtU, in_V, Vtarget, mu, maxiter=500, delta=0.01, normalize=False, nonzero=False):
    """hals_coupling_nnls_acc with V in the working dtype (parafac2)."""
    dt = L.resolve_dtype(UtM, UtU, in_V, Vtarget)
    b = L.to_device(UtM, dt)
    r, n = b.shape
    G_host = np.array(UtU.detach().cpu().numpy() if isinstance(UtU, torch.Tensor) else UtU, dtype=np.float64, copy=True)
    diag = np.diagonal(G_host)[:r].copy()
    idx = np.arange(r)
    G_host[idx, idx] = np.where(diag != 0, diag + float(mu), 0.0)          # nnls.py:316: test on UtU[k,k], divide by UtU[k,k] + mu
    G = L.to_device(G_host, dt)
    Vt = L.to_device(Vtarget, dt)
    if not np.prod(np.shape(in_V)):                                        # nnls.py:292-298 (start from the uncoupled least squares)
        G0 = L.to_device(UtU, dt)
        V = torch.linalg.solve(G0[:r, :r].double(), b.double())
        V.clamp_(min=0)
        scale = (b.double() * V).sum() / (G0[:r, :r].double() * (V @ V.T)).sum()
        V = (V * scale).to(dt).contiguous()
    else:
        V = L.to_device(in_V, dt)
        if V.data_ptr() == (in_V.data_ptr() if isinstance(in_V, torch.Tensor) else 0):
            V = V.clone()
    rhs = ops.axpby(1.0, b, float(mu), Vt[:r].contiguous())               # UtM + mu Vtarget
    res = hals_nnls_device(rhs, G, V, r, maxiter, delta, None, normalize, nonzero).cpu().numpy()
    if res[2] >= 0:
        raise ValueError("Column " + str(int(res[2])) + " is zero with nonzero condition")    # nnls.py:330
    out = V if isinstance(in_V, torch.Tensor) else V.cpu().numpy()
    return out, np.float64(res[0]), int(res[1]), _RHO_UNUSED
