"""Column-sharded NMF over several GPUs, one process per GPU (new: the reference is single-process).

Rank p of the torch.distributed group holds the column block X_p (m x n_p) of the data and the matching
block V_p (r x n_p) of the second factor; U (m x r) is replicated.  The arithmetic per block is the
one of nn_fac.nmf.compute_nmf (nmf.py:283-329); the exchange steps are described in nn_fac/_fast.py.
fp32; update_rule "hals" and "mu" with beta = 2 up to rank 128, "mu" with beta = 1 up to rank 64 (the tcgen05 path).
"""
import numpy as np
import torch

from nn_fac import _fast
from nn_fac.nmf import _check_step_arguments


def column_block(n, world, rank, align=128):
    """[lo, hi) of the columns owned by `rank`: equal blocks aligned to `align` columns (the last may be short)."""
    chunk = -(-n // world)
    chunk = -(-chunk // align) * align
    lo = min(rank * chunk, n)
    return lo, min(lo + chunk, n)


def compute_nmf_sharded(data_block, rank, U_in, V_block, n_iter_max=100, tol=1e-8, update_rule="hals", beta=2,
                        sparsity_coefficients=[None, None], fixed_modes=[], normalize=[False, False],
                        verbose=False, return_costs=False, group=None):
    """compute_nmf on this rank's column block.  Returns (U, V_block) or (U, V_block, cost_fct_vals, toc):
    U and the costs are identical on every rank, V_block is this rank's columns of V."""
    _check_step_arguments(update_rule, beta, sparsity_coefficients)
    if _fast.general_beta(update_rule, beta):
        raise NotImplementedError(f"the sharded path covers update_rule 'mu' with beta = 1 or 2 only (got beta = {beta})")
    if _fast.planes_of_precision() == 3:
        raise NotImplementedError("precision 'fp32x3' is not covered by the sharded path (its exchanges write two planes)")
    if not _fast.eligible(torch.float32, int(np.shape(U_in)[1]), update_rule, beta):
        raise NotImplementedError("the sharded path covers update_rule 'hals' and 'mu' with beta = 2 (rank <= 128) and 'mu' with "
                                  "beta = 1 (rank <= 64)")
    if group is None and torch.distributed.is_available() and torch.distributed.is_initialized():
        group = torch.distributed.group.WORLD
    state = _fast.FusedNMF(data_block, U_in, V_block, group=group)
    costs, toc = state.run(n_iter_max, tol, update_rule, sparsity_coefficients, fixed_modes, normalize, verbose, beta=beta)
    U_dev, V_dev = state.factors()
    as_out = (lambda t: t) if isinstance(data_block, torch.Tensor) else (lambda t: t.cpu().numpy())
    if return_costs:
        return as_out(U_dev), as_out(V_dev), costs, toc
    return as_out(U_dev), as_out(V_dev)
