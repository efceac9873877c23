"""Nonnegative matrix factorisation, B200 path (reference: nn_fac/nmf.py).

Same public functions and return conventions as the reference (``nmf``, ``compute_nmf``,
``one_nmf_step``); the body of ``one_nmf_step`` -- Gram / cross-product formation, the HALS solve
or multiplicative update, and the cost -- runs on the GPU.  ``compute_nmf`` uploads the data once
and keeps X and both factors resident for the whole outer loop; per iteration only the cost
scalars come back to the host (the reference's stop test ``|dcost| < tol`` needs them).

HALS always uses the deterministic inner stopping rule (the reference's ``deterministic=True``
semantics, nmf.py:414-416); the wall-clock rule is not reproducible and is not implemented.
"""
import time
import warnings

import numpy as np
import torch

import nn_fac.update_rules.mu as mu
import nn_fac.update_rules.nnls as nnls
import nn_fac.utils.errors as err
import nn_fac.utils.initialize_factors as init_factors
from nn_fac import _fast
from nn_fac import _lib as L
from nn_fac import _ops as ops


def nmf(data, rank, init="random", U_0=None, V_0=None, n_iter_max=100, tol=1e-8,
        update_rule="hals", beta=2,
        sparsity_coefficients=[None, None], fixed_modes=[], normalize=[False, False],
        verbose=False, return_costs=False, deterministic=False, seed=0):
    """Factorise `data` (m x n, nonnegative) as U V with U m x rank and V rank x n.

    Arguments, defaults, errors and returns follow nn_fac.nmf.nmf (nmf.py:19-193):
    returns (U, V) or, with return_costs, (U, V, cost_fct_vals, toc).
    update_rule "hals" minimises ||data - UV||_F^2 (+ 2*sparsity*||.||_1); "mu" the beta-divergence.
    """
    if min(data.shape) < rank:                                             # nmf.py:175-178
        rank = min(data.shape)
        warnings.warn(f"The rank is too high for the input matrix. It was set to {rank} instead.")
    if deterministic:
        np.random.seed(seed)                                               # nmf.py:180-181
    if init.lower() == "custom":
        if U_0 is None or V_0 is None:
            raise err.CustomNotValidFactors("Custom initialization, but (at least) one factor is set to 'None'")
    else:
        host = data.detach().cpu().numpy() if isinstance(data, torch.Tensor) else data
        U_0, V_0 = init_factors.nmf_initialization(host, rank, init, deterministic=deterministic, seed=seed)
    return compute_nmf(data, rank, U_0, V_0, n_iter_max=n_iter_max, tol=tol, update_rule=update_rule, beta=beta,
                       sparsity_coefficients=sparsity_coefficients, fixed_modes=fixed_modes, normalize=normalize,
                       verbose=verbose, return_costs=return_costs, deterministic=deterministic)


def _check_step_arguments(update_rule, beta, sparsity_coefficients):
    if update_rule not in ("hals", "mu"):                                  # nmf.py:387-390
        raise err.InvalidArgumentValue(f"Invalid update rule: {update_rule}") from None
    if update_rule == "hals" and beta != 2:
        raise err.InvalidArgumentValue(
            "The hals is only valid for the frobenius norm, corresponding to the beta divergence with beta = 2. "
            f"Here, beta was set to {beta}. To compute NMF with this value of beta, please use the mu update_rule."
        ) from None
    if len(sparsity_coefficients) != 2:                                    # nmf.py:392-393
        raise ValueError("NMF needs 2 sparsity coefficients to be performed")


class _Phase:
    """Optional CUDA-event bracket around one phase of an iteration (enabled by setting state.events = [])."""

    def __init__(self, state, name):
        self.state, self.name = state, name

    def __enter__(self):
        if self.state.events is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if self.state.events is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            self.state.events.append((self.name, self.e0, e1))


class DeviceNMF:
    """X, U (m x r), U^T (r x m) and V (r x n) resident on one GPU; one call = one outer iteration."""
    events = None

    def __init__(self, data, U, V, dtype, device=None):
        self.dtype = dtype
        self.X = L.to_device(data, dtype, device)
        self.U = L.to_device(U, dtype, device)
        self.V = L.to_device(V, dtype, device)
        if self.V.data_ptr() == (V.data_ptr() if isinstance(V, torch.Tensor) else 0):
            self.V = self.V.clone()
        self.m, self.n = self.X.shape
        self.r = self.U.shape[1]
        self.scal = torch.zeros(8, dtype=torch.float64, device=self.X.device)
        # fp32: X also lives as bf16 hi/lo planes in both orientations for the tcgen05 X passes
        self.plan = ops.NMFPlan(self.X).bind_rank(self.r) if (dtype == torch.float32 and self.r <= 128) else None
        self.hals_stats = torch.zeros((2, 4), dtype=torch.float64, device=self.X.device)

    # -- HALS -----------------------------------------------------------------------------------
    def hals_iteration(self, sparsity, fixed_modes, normalize):
        X, m, n, r = self.X, self.m, self.n, self.r
        if 0 not in fixed_modes:
            V = self.V
            with _Phase(self, "cross_U"):
                VVt = ops.gemm(V, (n, 1), V, (1, n), r, r, n)              # nmf.py:407
                if self.plan is not None:
                    VMt = self.plan.cross(0, V)                            # nmf.py:408 on tcgen05
                else:
                    VMt = ops.gemm(V, (n, 1), X, (1, n), r, m, n)          # nmf.py:408 (V X^T, r x m)
            with _Phase(self, "sweep_U"):
                Ut = ops.transpose(self.U)
                nnls.hals_nnls_device(VMt, VVt, Ut, r, maxiter=100, delta=0.01, sparsity_coefficient=sparsity[0],
                                      normalize=normalize[0], nonzero=False, result=self.hals_stats[0])  # nmf.py:415
                self.U = ops.transpose(Ut)
            self.Ut = Ut
        else:
            self.Ut = ops.transpose(self.U)
        if 1 not in fixed_modes:
            Ut = self.Ut
            with _Phase(self, "cross_V"):
                UtU = ops.gemm(Ut, (m, 1), Ut, (1, m), r, r, m)            # nmf.py:432
                if self.plan is not None:
                    UtM = self.plan.cross(1, Ut)                           # nmf.py:433 on tcgen05
                else:
                    UtM = ops.gemm(Ut, (m, 1), X, (n, 1), r, n, m)         # nmf.py:433
            with _Phase(self, "sweep_V"):
                nnls.hals_nnls_device(UtM, UtU, self.V, r, maxiter=100, delta=0.01, sparsity_coefficient=sparsity[1],
                                      normalize=normalize[1], nonzero=False, result=self.hals_stats[1])  # nmf.py:440
        # cost (nmf.py:449-452)
        with _Phase(self, "cost"):
            K = ops.matmul(self.U, self.V)
            ops.sq_diff(X, K, out=self.scal[0:1])
        sp = [0.0 if s is None else float(s) for s in sparsity]
        if sp[0] != 0.0 or sp[1] != 0.0:
            n1u = ops.norm1(self.U)
            n1v = ops.norm1(self.V)
            host = torch.cat([self.scal[0:1], n1u, n1v]).cpu().numpy()
            return float(host[0] + 2 * (sp[0] * host[1] + sp[1] * host[2]))
        return float(self.scal[0:1].cpu().numpy()[0])

    # -- MU ---------------------------------------------------------------------------------------
    def mu_iteration(self, beta, fixed_modes):
        if 0 not in fixed_modes:
            with _Phase(self, "update_U"):
                self.U = mu.mu_update_device(self.U, self.V, self.X, beta, "U")  # nmf.py:422
        if 1 not in fixed_modes:
            with _Phase(self, "update_V"):
                self.V = mu.mu_update_device(self.V, self.U, self.X, beta, "V")  # nmf.py:447
        with _Phase(self, "cost"):
            K = ops.matmul(self.U, self.V)
            ops.beta_divergence(self.X, K, beta, out=self.scal[0:1])         # nmf.py:455
        return float(self.scal[0:1].cpu().numpy()[0])

    def step(self, update_rule, beta, sparsity, fixed_modes, normalize):
        if update_rule == "hals":
            return self.hals_iteration(sparsity, fixed_modes, normalize)
        return self.mu_iteration(beta, fixed_modes)


def _to_output(t, like, dtype=None):
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)                               # small float32 problems compute in float64 (nn_fac/config.py)
    return t if isinstance(like, torch.Tensor) else t.cpu().numpy()


def compute_nmf(data, rank, U_in, V_in, n_iter_max=100, tol=1e-8,
                update_rule="hals", beta=2,
                sparsity_coefficients=[None, None], fixed_modes=[], normalize=[False, False],
                verbose=False, return_costs=False, deterministic=False):
    """Outer alternating loop (nmf.py:196-329): stops when |cost[-2] - cost[-1]| < tol."""
    if sparsity_coefficients is None:
        sparsity_coefficients = [None, None]
    if fixed_modes is None:
        fixed_modes = []
    if normalize is None or normalize is False:
        normalize = [False, False]
    dt, dt_out = L.working_dtype(int(np.prod(np.shape(data))), data, U_in, V_in)
    planes = _fast.planes_of_precision()
    if n_iter_max > 0 and _fast.eligible(torch.float32 if planes == 3 else dt, int(np.shape(U_in)[1]), update_rule, beta, planes=planes):
        # fp32, rank <= 64: two X passes per iteration on tcgen05, cost fused with a lag of one pass ("fp32x3": 3-plane plan)
        _check_step_arguments(update_rule, beta, sparsity_coefficients)
        fast = _fast.FusedNMF(data, U_in, V_in)
        cost_fct_vals, toc = fast.run(n_iter_max, tol, update_rule, sparsity_coefficients, fixed_modes, normalize, verbose,
                                      beta=beta)
        U_dev, V_dev = fast.factors()
        U_out, V_out = _to_output(U_dev, data, dt_out), _to_output(V_dev, data, dt_out)
        if return_costs:
            return U_out, V_out, cost_fct_vals, toc
        return U_out, V_out
    state = None
    cost_fct_vals, toc = [], []
    tic = time.time()
    for iteration in range(n_iter_max):
        _check_step_arguments(update_rule, beta, sparsity_coefficients)
        if state is None:
            state = DeviceNMF(data, U_in, V_in, dt)
        cost = state.step(update_rule, beta, sparsity_coefficients, fixed_modes, normalize)
        toc.append(time.time() - tic)
        cost_fct_vals.append(cost)
        if verbose:
            if iteration == 0:
                print('Normalized cost function value={}'.format(cost))
            else:
                gain = cost_fct_vals[-2] - cost_fct_vals[-1]
                line = 'Normalized cost function value={}, variation={}.'.format(cost_fct_vals[-1], gain)
                print(line if gain > 0 else '\033[91m' + line + '\033[0m')
        if iteration > 0 and abs(cost_fct_vals[-2] - cost_fct_vals[-1]) < tol:   # nmf.py:320
            if verbose:
                print('Converged in {} iterations.'.format(iteration))
            break
    if state is None:
        U_out, V_out = np.array(U_in), np.array(V_in)
    else:
        U_out, V_out = _to_output(state.U, data, dt_out), _to_output(state.V, data, dt_out)
    if return_costs:
        return U_out, V_out, cost_fct_vals, toc
    return U_out, V_out


def one_nmf_step(data, rank, U_in, V_in, norm_data, update_rule, beta,
                 sparsity_coefficients, fixed_modes, normalize, deterministic):
    """One U update, one V update and the cost (nmf.py:332-458).  Inputs are not modified.

    Host arrays are uploaded on every call; use compute_nmf / nmf to keep the data resident.
    `norm_data` and `deterministic` are accepted for signature parity (the cost is not normalised,
    nmf.py:457, and the inner stop rule is always the deterministic one).
    """
    _check_step_arguments(update_rule, beta, sparsity_coefficients)
    dt, dt_out = L.working_dtype(int(np.prod(np.shape(data))), data, U_in, V_in)
    state = DeviceNMF(data, U_in, V_in, dt)
    cost = state.step(update_rule, beta, sparsity_coefficients, fixed_modes, normalize)
    return _to_output(state.U, data, dt_out), _to_output(state.V, data, dt_out), cost
