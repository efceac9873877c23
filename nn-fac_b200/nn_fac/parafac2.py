"""Nonnegative PARAFAC2 with flexible coupling, B200 path (reference: nn_fac/parafac2.py, SURVEY.md 8(f) row N4).

Same functions and return conventions as the reference (``parafac_2``, ``compute_parafac_2``, ``one_step_parafac2``,
``compute_P_k``, ``compute_W_star``).  Every product that touches a slice of the data and every NNLS solve -- the coupled
solve ``hals_coupling_nnls_acc`` for the W_k (parafac2.py:522), the plain ``hals_nnls_acc`` for the diagonals D_k (:548) and
for H (:581) -- runs on the GPU through libnnfac_b200; the rank x rank bookkeeping and the r x r SVDs of ``compute_P_k``
(:610) stay on the host like in the reference.  The slices are uploaded once per ``compute_parafac_2`` call.

As everywhere in this package the inner solves use the deterministic stop rule (the reference passes its wall-clock rule
``alpha=0.5, atime=timer`` here: parafac2.py:522-524, :548, :581); parity is defined against the reference run with
``alpha=inf`` (tests/golden/make_golden.py::parafac2_cases).  Quirks that are kept because callers see them: ``parafac_2``
ignores its ``normalize``, ``tol_mu`` and ``step_mu`` arguments when it calls ``compute_parafac_2`` (parafac2.py:198-200),
``one_step_parafac2`` refreshes P_k only ``if 4 in fixed_modes`` (:497) and W* only ``if 3 in fixed_modes`` (:503), and
W* of the "nndsvd" start is divided by ``nb_channel - 1`` (initialize_factors.py:155).  Two defects are not reproduced: the
reference's "nndsvd" initialiser forgets its ``return`` (initialize_factors.py:139-156), and ``err.InitializationNotValid``
(parafac2.py:322) does not exist in utils/errors.py -- here that case raises ``err.InvalidInitializationType``.
"""
import time

import numpy as np
import torch

import nn_fac.update_rules.nnls as nnls
import nn_fac.utils.errors as err
import nn_fac.utils.initialize_factors as init_factors
from nn_fac import _lib as L
from nn_fac import _ops as ops


def parafac_2(tensor_slices, rank, init_with_P, init="random", W_list_in=None, H=None, D_list_in=None, W_star=None, P_list=None,
              tol_mu=1e6, step_mu=1.02, n_iter_max=100, tol=1e-6,
              sparsity_coefficient=None, fixed_modes=[], normalize=[False, False, False, False, False],
              verbose=False, return_costs=False, deterministic=False, seed=0):
    """parafac2.py:18-200.  Returns (W_list, H, D_list) or, with return_costs, (W_list, H, D_list, cost_fct_vals, toc)."""
    if deterministic:
        np.random.seed(seed)
    if init.lower() == "custom":
        if W_list_in is None or H is None or D_list_in is None:
            raise err.CustomNotValidFactors("Custom initialization, but (at least) one factor is set to 'None'")
        W_list, D_list = W_list_in.copy(), D_list_in.copy()
    else:
        W_list, H, D_list, P_list, W_star = init_factors.parafac2_initialization(tensor_slices, rank, init, init_with_P,
                                                                                 deterministic=deterministic, seed=seed)
    return compute_parafac_2(tensor_slices, rank, W_list_in=W_list, H_0=H, D_list_in=D_list, init_with_P=init_with_P,
                             W_star_in=W_star, P_list_in=P_list, n_iter_max=n_iter_max, tol=tol,
                             sparsity_coefficient=sparsity_coefficient, fixed_modes=fixed_modes,
                             normalize=[False, False, False, False], verbose=verbose, return_costs=return_costs)   # sic, :198-200


def _fro(a):
    return np.linalg.norm(a, ord='fro')


class _Slices:
    """The data slices resident on the GPU, with the products the updates need (each one pass over a slice)."""

    def __init__(self, tensor_slices):
        self.host = tensor_slices
        dt = L.resolve_dtype(*tensor_slices)
        self.dtype = dt
        self.dev = [L.to_device(s, dt) for s in tensor_slices]

    def up(self, a):
        return L.to_device(np.ascontiguousarray(a), self.dtype)

    def right(self, k, A):
        """A (q x n) -> A X_k^T (q x r): VMt of the W_k update (parafac2.py:517)."""
        X = self.dev[k]
        return ops.matmul(self.up(A), X.T)

    def left(self, k, A):
        """A (r x q) -> A^T X_k (q x n): the D_k and H updates (:535, :576)."""
        X = self.dev[k]
        return ops.matmul(self.up(A).T, X)

    def residual_sq(self, k, A, B):
        """||X_k - A B||_F^2 (:329, :342, :593)."""
        K = ops.matmul(self.up(A), self.up(B))
        return float(ops.sq_diff(self.dev[k], K).item())


def compute_parafac_2(tensor_slices, rank, W_list_in, H_0, D_list_in, init_with_P, W_star_in=None, P_list_in=None,
                      tol_mu=1e6, step_mu=1.02, n_iter_max=100, tol=1e-8,
                      sparsity_coefficient=None, fixed_modes=[], normalize=[False, False, False, False, False],
                      verbose=False, return_costs=False):
    """Outer loop of parafac2.py:202-400 (mu schedule of :340-349 included)."""
    nb_channel = len(tensor_slices)
    W_list = W_list_in.copy()
    H = H_0.copy()
    D_list = D_list_in.copy()
    W_star = None if W_star_in is None else W_star_in.copy()
    P_list = None if P_list_in is None else P_list_in.copy()
    if W_star is None and P_list is None:
        raise err.InvalidInitializationType("Initialization not valid: W^* and P_list cannot be both None.")
    slices = _Slices(tensor_slices)
    cost_fct_vals, toc, norm_slices, couple_error, couple_errors = [], [], [], [], []
    tic = time.time()
    increasing_mu = True
    mu_list = np.zeros(nb_channel)
    for k in range(nb_channel):                                            # :328-333
        mu_list[k] = slices.residual_sq(k, W_list[k] @ D_list[k], H) / (10 * _fro(W_list[k]) ** 2)
        norm_slices.append(np.sqrt(float(ops.sq_diff(slices.dev[k]).item())))
    for iteration in range(n_iter_max):
        previous_cost_fct_val = None if iteration == 0 else cost_fct_vals[-1]
        if iteration == 1:                                                 # :342-344
            for k in range(nb_channel):
                mu_list[k] = 0.2 * np.sqrt(slices.residual_sq(k, W_list[k] @ D_list[k], H)) / couple_error[k]
        if iteration == 2:
            increasing_mu = True
        W_list, H, D_list, W_star, P_list, mu_list, cost, couple_error, increasing_mu = _one_step(
            slices, rank, W_list, H, D_list, mu_list, norm_slices, previous_cost_fct_val, increasing_mu=increasing_mu,
            init_with_P=init_with_P, P_list_in=P_list, W_star_in=W_star, sparsity_coefficient=sparsity_coefficient,
            fixed_modes=fixed_modes, normalize=normalize)
        toc.append(time.time() - tic)
        cost_fct_vals.append(cost)
        couple_errors.append(couple_error)
        if verbose:
            if iteration == 0:
                print('Normalized cost function value={}'.format(cost))
                for k in range(nb_channel):
                    print('Couple_error for channel {} = {}'.format(k, couple_errors[iteration][k]))
            else:
                gain = cost_fct_vals[-2] - cost_fct_vals[-1]
                line = 'Normalized cost function value={}, variation={}.'.format(cost_fct_vals[-1], gain)
                print(line if gain > 0 else '\033[91m' + line + '\033[0m')
                for k in range(nb_channel):
                    gain = couple_errors[-2][k] - couple_errors[-1][k]
                    line = 'Couple_error for channel {} = {}, variation={}.'.format(k, couple_errors[-1][k], gain)
                    print(line if gain > 0 else '\033[91m' + line + '\033[0m')
        if iteration > 0 and abs(cost_fct_vals[-2] - cost_fct_vals[-1]) < tol:
            if verbose:
                print('Converged in {} iterations.'.format(iteration))
            break
    W_list, H, D_list = _as_output(W_list), L.as_output(np.array(H)), _as_output(D_list)
    if return_costs:
        return W_list, H, D_list, cost_fct_vals, toc
    return W_list, H, D_list


def _as_output(arrays):
    """L.as_output over a list of arrays (or a stacked array, which normalize[2] makes of D_list)."""
    return L.as_output(arrays) if isinstance(arrays, np.ndarray) else [L.as_output(a) for a in arrays]


def one_step_parafac2(slices, rank, W_list_in, H_in, D_list_in, mu_list_in, norm_slices,
                      previous_cost_fct_val, increasing_mu=True, tol_mu=1e6, step_mu=1.02,
                      init_with_P=True, W_star_in=None, P_list_in=None,
                      sparsity_coefficient=None, fixed_modes=[], normalize=[False, False, False, False, False]):
    """One pass over all channels (parafac2.py:402-602).  The slices are uploaded on every call; use compute_parafac_2 to
    keep them resident."""
    W_list, H, D_list, W_star, P_list, mu_list, cost, couple_error, increasing_mu = _one_step(
        _Slices(slices), rank, W_list_in, H_in, D_list_in, mu_list_in, norm_slices, previous_cost_fct_val,
        increasing_mu=increasing_mu, tol_mu=tol_mu, step_mu=step_mu, init_with_P=init_with_P, W_star_in=W_star_in,
        P_list_in=P_list_in, sparsity_coefficient=sparsity_coefficient, fixed_modes=fixed_modes, normalize=normalize)
    return (_as_output(W_list), L.as_output(H), _as_output(D_list), L.as_output(W_star), _as_output(P_list), mu_list, cost,
            couple_error, increasing_mu)


def _one_step(slices, rank, W_list_in, H_in, D_list_in, mu_list_in, norm_slices, previous_cost_fct_val, increasing_mu=True,
              tol_mu=1e6, step_mu=1.02, init_with_P=True, W_star_in=None, P_list_in=None, sparsity_coefficient=None,
              fixed_modes=[], normalize=[False, False, False, False, False]):
    W_list = W_list_in.copy()
    D_list = D_list_in.copy()
    H = H_in.copy()
    mu_list = mu_list_in.copy()
    cost_fct_val = 0
    nb_channel = len(W_list)
    if P_list_in is None and W_star_in is None:                           # :478-485
        raise ValueError('The list of P_k and W^* are both to None: one has to be set for the operation.')
    elif init_with_P == True and P_list_in is None:                       # noqa: E712
        raise ValueError('PARAFAC2 is set with the init of P_k, but they are set to None.')
    elif init_with_P == False and W_star_in is None:                      # noqa: E712
        raise ValueError('PARAFAC2 is set with the init of W^*, but it is set to None.')
    if init_with_P:                                                       # :488-498
        P_list = P_list_in.copy()
        W_star = compute_W_star(P_list, W_list, mu_list, nb_channel, normalize=True)
        if 4 in fixed_modes:
            P_list = compute_P_k(W_list, W_star, nb_channel)
    else:                                                                 # :500-505
        W_star = W_star_in
        P_list = compute_P_k(W_list, W_star, nb_channel)
        if 3 in fixed_modes:
            W_star = compute_W_star(P_list, W_list, mu_list, nb_channel, normalize=normalize[3])

    for k in range(nb_channel):
        if 0 not in fixed_modes:
            # W_k: coupled solve against P_k W*  (:509-524)
            DkH = D_list[k] @ H
            VVt = DkH @ DkH.T
            VMt = slices.right(k, DkH)                                    # DkH X_k^T on the GPU
            W_list[k] = np.transpose(nnls._hals_coupling_nnls_acc(VMt, VVt, np.transpose(W_list[k]), np.transpose(P_list[k] @ W_star),
                                                                 mu_list[k], maxiter=100, delta=0.01, normalize=normalize[0],
                                                                 nonzero=False)[0])
        if 2 not in fixed_modes:
            # D_k: the diagonal is an NNLS with the Khatri-Rao product of W_k and H^T as dictionary (:526-557).  Its Gram is the
            # Hadamard product of the Grams and its right-hand side the diagonal of W_k^T X_k H^T: the (r n) x rank
            # Khatri-Rao matrix of :531 is never formed.
            UtU = (W_list[k].T @ W_list[k]) * (H @ H.T)
            WtX = slices.left(k, W_list[k])                               # W_k^T X_k on the GPU
            UtM = ops.row_sums(ops.hadamard_(WtX, slices.up(H))).reshape(-1, 1).cpu().numpy()
            diag_D = np.reshape(np.diagonal(D_list[k]), (-1, 1))
            new_D = nnls._hals_nnls_acc(UtM, UtU, diag_D, maxiter=100, delta=0.01, sparsity_coefficient=None, normalize=False,
                                       nonzero=False)[0]
            D_list[k] = np.diag(np.asarray(new_D).flatten())
    if normalize[2]:                                                      # :559-565 (D_list must be an array here, as in the reference)
        D_list = np.array(D_list)
        for note_index in range(rank):
            norm = np.linalg.norm(D_list[:, note_index], ord='fro')
            if norm == 0:
                D_list[:, note_index, note_index] = [1 / (nb_channel ** 2) for k in range(nb_channel)]
            else:
                D_list[:, note_index] /= np.linalg.norm(D_list[:, note_index], ord='fro')

    if 1 not in fixed_modes:
        # H: stacked least squares over the channels (:567-582)
        UtU = np.zeros((rank, rank))
        UtM = None
        for k in range(nb_channel):
            WkDk = W_list[k] @ D_list[k]
            UtU += WkDk.T @ WkDk
            part = slices.left(k, WkDk)                                   # (W_k D_k)^T X_k on the GPU
            UtM = part if UtM is None else ops.axpby(1.0, UtM, 1.0, part)
        H = nnls._hals_nnls_acc(UtM, UtU, slices.up(H), maxiter=100, delta=0.01, sparsity_coefficient=sparsity_coefficient,
                               normalize=normalize[1], nonzero=False)[0].cpu().numpy()

    couple_error = []
    if sparsity_coefficient != None:                                      # noqa: E711
        cost_fct_val = sparsity_coefficient * np.linalg.norm(H, ord=1)
    for k in range(nb_channel):                                           # :589-600
        couple_error.append(_fro(W_list[k] - P_list[k] @ W_star))
        slice_rec_error = slices.residual_sq(k, W_list[k] @ D_list[k], H) + (mu_list[k] * couple_error[k] ** 2) / norm_slices[k]
        cost_fct_val += slice_rec_error
        if previous_cost_fct_val != None:                                 # noqa: E711
            if mu_list[k] < tol_mu and (previous_cost_fct_val - cost_fct_val) > 0 and increasing_mu:
                mu_list[k] *= step_mu
            elif increasing_mu:
                increasing_mu = False
    return W_list, H, D_list, W_star, P_list, mu_list, cost_fct_val, couple_error, increasing_mu


def compute_P_k(W_list, W_star, nb_channel):
    """parafac2.py:605-612: P_k = U V^T of the SVD of W_k W*^T (r x r, host)."""
    list_of_P = []
    nb_columns_P = W_star.shape[0]
    for k in range(nb_channel):
        U, S, Vt = np.linalg.svd(W_list[k] @ W_star.T)
        list_of_P.append(U[:, 0:nb_columns_P] @ Vt[0:nb_columns_P, :])
    return list_of_P


def compute_W_star(P_list, W_list, mu_list, nb_channel, normalize=False):
    """parafac2.py:614-630."""
    nb_columns = W_list[0].shape[1]
    nb_lines = P_list[0].shape[1]
    W_star_local_sum = np.zeros((nb_lines, nb_columns))
    for k in range(nb_channel):
        W_star_local_sum += mu_list[k] * P_list[k].T @ W_list[k]
    local_W_star = W_star_local_sum / np.sum(mu_list)
    if normalize:
        for index in range(nb_columns):
            norm = np.linalg.norm(local_W_star[:, index], ord=2)
            if norm != 0:
                local_W_star[:, index] /= norm
    return local_W_star
