"""beta-divergence multiplicative updates on the GPU (reference: nn_fac/update_rules/mu.py).

fp64 mode (and any shape the tensor-core kernels do not cover) follows the reference literally:
K = U V is formed, the element-wise terms K^(beta-2)*M and K^(beta-1) are applied, and the two
contractions against the other factor run on the library's strided GEMM.  The fp32 headline path
for NMF (nmf.py) uses the fused tcgen05 kernel instead, where K never reaches HBM.
"""
import numpy as np
import torch

import nn_fac.utils.errors as err
from nn_fac import _lib as L
from nn_fac import _ops as ops
from nn_fac.utils.beta_divergence import gamma_beta

epsilon = 1e-12  # mu.py:18


def mu_update_device(F, other, X, beta, which, K=None):
    """One multiplicative update of F on device tensors, without transposed copies.

    which == "U": F is U (m x r), other is V (r x n)   -> mu.py:82-97 as written.
    which == "V": F is V (r x n), other is U (m x r)   -> the transposed call of mu.py:27.
    K: optional precomputed U V (m x n); it is overwritten.
    """
    U, V = (F, other) if which == "U" else (other, F)
    m, r = U.shape
    n = V.shape[1]
    if K is None:
        K = ops.matmul(U, V)                                               # mu.py:82
    g = gamma_beta(beta)
    if beta == 2:
        P, Q = X, K                                                        # mu.py:89-91
    elif beta == 1:
        P, Q = ops.mu_terms(K, X, beta, want_q=False, out_p=K)[0], None    # mu.py:84 (K**-1 * M, in place)
    else:
        P, Q = ops.mu_terms(K, X, beta, want_q=True, out_p=torch.empty_like(K), out_q=K)
    if which == "U":
        num = ops.gemm(P, (n, 1), V, (1, n), m, r, n)                      # (.) @ V.T
        if Q is None:
            return ops.mu_apply(U, num, den_vec=ops.row_sums(V), vec_per_row=False, gamma=g, floor=epsilon)
        den = ops.gemm(Q, (n, 1), V, (1, n), m, r, n)
        return ops.mu_apply(U, num, den_mat=den, gamma=g, floor=epsilon)
    num = ops.gemm(U, (1, r), P, (n, 1), r, n, m)                          # U.T @ (.)
    if Q is None:
        col_sums = ops.row_sums(ops.transpose(U))
        return ops.mu_apply(V, num, den_vec=col_sums, vec_per_row=True, gamma=g, floor=epsilon)
    den = ops.gemm(U, (1, r), Q, (n, 1), r, n, m)
    return ops.mu_apply(V, num, den_mat=den, gamma=g, floor=epsilon)


def _out(t, like):
    t = L.as_output(t)
    return t if isinstance(like, torch.Tensor) else t.cpu().numpy()


def switch_alternate_mu(data, U, V, beta, matrix):
    """mu.py:20-29: update U ("U"/"W") or V ("V"/"H")."""
    if matrix not in ("U", "W", "V", "H"):
        raise err.InvalidArgumentValue(
            f"Invalid value for matrix: got {matrix}, but it must be 'U' or 'W' for the first matrix, "
            "and 'V' or 'H' for the second one.") from None
    if beta < 0:
        raise err.InvalidArgumentValue("Invalid value for beta: negative one.") from None
    dt = L.resolve_dtype(data, U, V)
    Xd, Ud, Vd = L.to_device(data, dt), L.to_device(U, dt), L.to_device(V, dt)
    if matrix in ("U", "W"):
        return _out(mu_update_device(Ud, Vd, Xd, beta, "U"), U)
    return _out(mu_update_device(Vd, Ud, Xd, beta, "V"), V)


def mu_betadivmin(U, V, M, beta):
    """mu.py:31-97: U <- max(U * ((K^(beta-2) * M) V^T / (K^(beta-1) V^T))^gamma, 1e-12), K = U V."""
    if beta < 0:
        raise err.InvalidArgumentValue("Invalid value for beta: negative one.") from None
    dt = L.resolve_dtype(U, V, M)
    return _out(mu_update_device(L.to_device(U, dt), L.to_device(V, dt), L.to_device(M, dt), beta, "U"), U)


def _ones_contracted(factors):
    """ones x_n F_n^T (mu.py:144, 159 for beta = 1) in closed form: the outer product of the factors' column sums.  The
    reference contracts a tensor of ones of the size of the data through every mode for it."""
    dn = None
    for mode, F in enumerate(factors):
        s = ops.row_sums(ops.transpose(F))                                 # column sums of F_n (r_n)
        shape = [1] * len(factors)
        shape[mode] = s.shape[0]
        dn = s.reshape(shape) if dn is None else dn * s.reshape(shape)
    return dn.contiguous()


def mu_tensorial_device(G, factors, T, beta, plan0=None):
    """Tucker-core multiplicative update on device tensors (mu.py:138-159).

    plan0 (beta = 1, fp32, ranks <= 64): the NMF plan of unfold(T, 0).  The first contraction of the numerator,
    F_0^T unfold(T / K, 0), is then the V-side numerator of one fused tcgen05 pass over the planes of that unfolding
    with U = F_0 and V = unfold(G x_{j>0} F_j, 0): neither K nor T / K is ever written."""
    if beta == 1 and plan0 is not None:
        B0 = ops.multi_mode_dot(G, factors, skip=0)                         # r_0 x I_1 x ... (K = F_0 x_0 B0, mu.py:141)
        plan0.set_factor(0, ops.transpose(factors[0]))
        plan0.set_factor(1, B0.reshape(B0.shape[0], -1))
        P, _ = plan0.fused(1, 1, want_cost=False)                           # F_0^T unfold(T / K, 0): r_0 x (I_1 ...)
        up = ops.multi_mode_dot(P.reshape(B0.shape), factors, skip=0, transpose=True)
        dn = _ones_contracted(factors)
        return ops.mu_apply(G.reshape(G.shape[0], -1), up.reshape(G.shape[0], -1), den_mat=dn.reshape(G.shape[0], -1),
                            gamma=gamma_beta(beta), floor=epsilon).reshape(G.shape)
    K = ops.multi_mode_dot(G, factors)                                     # mu.py:141
    if beta == 2:
        L2, L1 = T, K
    elif beta == 1:
        L2 = ops.mu_terms(K, T, beta, want_q=False, out_p=K)[0]
        L1 = None                                                          # mu.py:144 (np.ones): closed form below
    else:
        L2, L1 = ops.mu_terms(K, T, beta, want_q=True, out_p=torch.empty_like(K), out_q=K)
    up = ops.multi_mode_dot(L2, factors, transpose=True)
    dn = ops.multi_mode_dot(L1, factors, transpose=True) if L1 is not None else _ones_contracted(factors)
    return ops.mu_apply(G.reshape(G.shape[0], -1), up.reshape(G.shape[0], -1), den_mat=dn.reshape(G.shape[0], -1),
                        gamma=gamma_beta(beta), floor=epsilon).reshape(G.shape)


def mu_tensorial(G, factors, tensor, beta):
    """mu.py:99-159."""
    if beta < 0:
        raise err.InvalidArgumentValue("Invalid value for beta: negative one.") from None
    dt = L.resolve_dtype(G, tensor, *factors)
    out = mu_tensorial_device(L.to_device(G, dt), [L.to_device(f, dt) for f in factors], L.to_device(tensor, dt), beta)
    return _out(out, G)
