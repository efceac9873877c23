"""Nonnegative PARAFAC / CP (NTF), B200 path (reference: nn_fac/ntf.py).

``ntf`` / ``compute_ntf`` keep the tensor resident on the GPU; the per-mode MTTKRP contracts the
tensor in place through strided access (no unfolded copies: the reference makes one copy of the
tensor per mode, ntf.py:309-311).  HALS uses the deterministic inner stopping rule.

Reference quirk kept: ``ntf`` returns ``np.array(factors)`` (ntf.py:342-344), which numpy >= 1.24
rejects for non-cubic tensors; here a non-cubic result is returned as an object array of factors.
"""
import os
import time

import numpy as np
import torch

import nn_fac.update_rules.mu as mu
import nn_fac.update_rules.nnls as nnls
import nn_fac.utils.errors as err
import nn_fac.utils.initialize_factors as init_factors
from nn_fac import _lib as L
from nn_fac._graph import try_capture
from nn_fac import _ops as ops


def ntf(tensor, rank, init="random", factors_0=[], n_iter_max=100, tol=1e-8,
        update_rule="hals", beta=2,
        sparsity_coefficients=[], fixed_modes=[], normalize=[],
        verbose=False, return_costs=False):
    """Arguments, defaults and returns follow nn_fac.ntf.ntf (ntf.py:19-199)."""
    nb_modes = len(tensor.shape)
    if init.lower() == "custom":                                            # ntf.py:184-191
        factors = factors_0
        if len(factors) != nb_modes:
            raise err.CustomNotEngouhFactors("Custom initialization, but not enough factors")
        for array in factors:
            if array is None:
                raise err.CustomNotValidFactors("Custom initialization, but one factor is set to 'None'")
    else:
        host = tensor.detach().cpu().numpy() if isinstance(tensor, torch.Tensor) else tensor
        factors = init_factors.ntf_initialization(host, rank, init, deterministic=False, seed=0)   # ntf.py:194
    return compute_ntf(tensor, rank, factors, n_iter_max=n_iter_max, tol=tol, update_rule=update_rule, beta=beta,
                       sparsity_coefficients=sparsity_coefficients, fixed_modes=fixed_modes, normalize=normalize,
                       verbose=verbose, return_costs=return_costs)


def _check_step_arguments(update_rule, beta):
    if update_rule not in ("hals", "mu"):                                   # ntf.py:422-425
        raise err.InvalidArgumentValue(f"Invalid update rule: {update_rule}") from None
    if update_rule == "hals" and beta != 2:
        raise err.InvalidArgumentValue(
            "The hals is only valid for the frobenius norm, corresponding to the beta divergence with beta = 2. "
            f"Here, beta was set to {beta}. To compute NMF with this value of beta, please use the mu update_rule."
        ) from None


class DeviceNTF:
    """Tensor (C order) and factors resident on one GPU."""

    def __init__(self, tensor, factors, dtype, device=None):
        self.T = L.to_device(tensor, dtype, device)
        self.shape = tuple(self.T.shape)
        self.factors = [L.to_device(f, dtype, device) for f in factors]
        self.factors_t = [ops.transpose(f) for f in self.factors]           # rank-major copies (r x I): sweep / Gram / MTTKRP layout
        self.norm_sq = None
        self._grams, self._gram_ok = None, [False] * len(self.factors)      # see _gram
        self.stats = torch.zeros(4, dtype=torch.float64, device=self.T.device)
        # fp32, rank <= 128: the MTTKRP of every mode runs on tcgen05 over ONE copy of the tensor as bf16 hi/lo planes (4 bytes
        # per element, what the fp32 tensor itself takes): mode 0 reads them as the rows of unfold(T, 0); the last mode reads the
        # same planes as an MN-major operand, middle modes through a 3-D TMA map (NMFPlan.view) -- the reference copies the
        # tensor once per mode (ntf.py:309-311).  Extents that cannot be addressed in place (trailing extent not a multiple of
        # 64 for a middle mode, ...) get a one-sided plan on a copy of that unfolding; not enough memory for the planes at all:
        # the strided CUDA-core MTTKRP on the tensor itself (self.plans None).
        self.plans = None
        rank = int(self.factors[0].shape[1])
        if dtype == torch.float32 and rank <= 128 and self.T.dim() >= 2 and os.environ.get("NNFAC_NTF_TC", "1") != "0":
            try:
                nm = self.T.dim()
                base = ops.NMFPlan(self.T.reshape(self.shape[0], -1)).bind_rank(rank, sides=1)
                self.plans = [base]
                for mode in range(1, nm):
                    left, I, right = ops._split(list(self.shape), mode)
                    view = base.view(left, I, right, rank) if os.environ.get("NNFAC_NTF_VIEWS", "1") != "0" else None
                    if view is None:
                        Xm = self.T.movedim(mode, 0).reshape(self.shape[mode], -1).contiguous()
                        view = ops.NMFPlan(Xm).bind_rank(rank, sides=1)
                        del Xm
                    self.plans.append(view)
            except torch.cuda.OutOfMemoryError:
                self.plans = None
                torch.cuda.empty_cache()

    def direct_cost(self, update_rule, fixed_modes=()):
        """fp32 on a 3-way tensor with plans (HALS; MU at rank <= 64, see _mu_pass): the objective is formed on chip by a fused
        pass over the tensor, for the state the iteration started from.

        HALS: the objective is the DIRECT residual ||T - [[A, B, C]]||^2 of the state an
        iteration starts from, formed on chip by the fused pass that also yields the first MTTKRP of that iteration (the model
        tile never reaches HBM) -- instead of the reference's ||T||^2 - 2 <F, rhs> + ||F krao^T||^2 (ntf.py:470), which
        subtracts numbers of the size of ||T||^2 and in fp32 keeps an error of ~7e-7 ||T||^2 (the truncation of the tensor
        core's fp32 accumulator biases rhs by -3.5e-7): 1.4e-4 of the objective at C4, more when the fit is better.
        The pass runs on the plan of the first free mode when that is a full plan; when it is a view (mode 0 fixed), on the
        plan of mode 0, which always is one: one extra pass over the tensor per iteration, its MTTKRP unused
        (_residual_mode)."""
        free = [m for m in range(len(self.shape)) if m not in fixed_modes]
        if self.plans is None or self.T.dim() != 3 or self.T.dtype != torch.float32 or not free:
            return False
        if update_rule == "mu":
            return int(self.factors[0].shape[1]) <= 64
        return update_rule == "hals" and os.environ.get("NNFAC_NTF_DIRECT", "1") != "0"

    def _residual_mode(self, fixed_modes):
        """The mode whose fused pass forms the direct residual (the fused pass needs a full plan, a view has no row planes):
        the first free mode, whose MTTKRP the pass also yields, or mode 0 when that one is a view."""
        free = [m for m in range(len(self.shape)) if m not in fixed_modes]
        return free[0] if free and getattr(self.plans[free[0]], "_base", None) is None else 0

    def _residual_pass(self, mode):
        """Fused pass over unfold(T, mode): returns ((unfold(T, mode) @ krao)^T, || T - F_mode krao^T ||^2) for the CURRENT factors."""
        others = [i for i in range(3) if i != mode]
        plan = self.plans[mode]
        plan.set_factor(0, self.factors_t[mode])
        plan.set_krao_rows(self.factors_t[others[0]], self.factors_t[others[1]])
        return plan.fused(0, 0)

    def _mu_pass(self, mode, beta, want_cost):
        """MU pass of the tensor core over unfold(T, mode) for the CURRENT factors (3-way tensor, rank <= 64, beta != 2): the model
        tile F_mode krao^T is formed on chip, never in HBM, and X is read once from the planes (views: in place).  The numerator
        partials (beta != 1: the denominator partials too) stay in the plan for _mu_finish; returns d_beta(T | [[F]]) as a device
        scalar when want_cost."""
        others = [i for i in range(3) if i != mode]
        plan = self.plans[mode]
        plan.set_factor_rows(self.factors_t[mode])
        plan.set_krao(self.factors_t[others[0]], self.factors_t[others[1]])
        if beta == 1:
            return plan.fused(0, 1, want_cost=want_cost, keep_partials=True)[1]
        return plan.fused_beta(0, beta, want_cost=want_cost)

    def _mu_finish(self, mode, beta):
        """The update of factor `mode` from its _mu_pass (mu.py:84-97); returns it rank-major (r x I)."""
        from nn_fac.utils.beta_divergence import gamma_beta
        plan = self.plans[mode]
        if beta == 1:
            # column sums of krao = colsum(F_a) * colsum(F_b)
            a, b = (self.factors_t[i] for i in range(3) if i != mode)
            den = ops.hadamard_(ops.row_sums(a), ops.row_sums(b))
            return plan.mu_finish_rows(self.factors_t[mode], mu.epsilon, den=den)
        return plan.mu_finish_rows(self.factors_t[mode], mu.epsilon, gamma=gamma_beta(beta))

    def _mu_cost_mode(self, beta, fixed_modes):
        """The mode whose pass forms the objective of an MU iteration: the first free mode (beta = 2: as for HALS)."""
        if beta == 2:
            return self._residual_mode(fixed_modes)
        return [m for m in range(len(self.shape)) if m not in fixed_modes][0]

    def cost_terms_now(self, sparsity, fixed_modes=(), update_rule="hals", beta=2):
        """Device vector [direct residual / beta-divergence of the current state, l1 norms for the sparsity terms...] (closing pass
        of a run)."""
        if update_rule == "mu" and beta != 2:
            res = self._mu_pass(self._mu_cost_mode(beta, fixed_modes), beta, True)
        else:
            _, res = self._residual_pass(self._residual_mode(fixed_modes))
        terms = [res]
        for idx, sp in enumerate(sparsity):
            if sp:
                terms.append(ops.norm1(self.factors[idx]))
        return torch.cat([t.reshape(1).to(torch.float64) for t in terms])

    def _gram(self, i):
        """F_i^T F_i of the HALS path, kept until factor i changes (the reference recomputes the Gram of every other factor
        for every mode, ntf.py:442-445: each one twice per iteration).  Fixed buffers, so that a graph-replayed iteration
        reads what the previous replay wrote."""
        if self._grams is None:
            r = int(self.factors_t[0].shape[0])
            self._grams = [torch.empty((r, r), dtype=self.T.dtype, device=self.T.device) for _ in self.factors_t]
        if not self._gram_ok[i]:
            ops.gram(self.factors_t[i], out=self._grams[i])
            self._gram_ok[i] = True
        return self._grams[i]

    def invalidate(self):
        """The factors were replaced from outside (roll-back of a speculative iteration)."""
        self._gram_ok = [False] * len(self.factors)

    def get_state(self):
        return list(self.factors) + list(self.factors_t)

    def set_state(self, tensors):
        k = len(tensors) // 2
        self.factors, self.factors_t = list(tensors[:k]), list(tensors[k:])

    def khatri_rao(self, skip):
        kept = [f for i, f in enumerate(self.factors) if i != skip]
        out = kept[0]
        for f in kept[1:]:
            out = ops.khatri_rao(out, f)                                    # ntf.py:448
        return out

    def mttkrp(self, mode, krao):
        """unfold(T, mode) @ krao without forming the unfolding (ntf.py:449)."""
        left, I, right = ops._split(list(self.shape), mode)
        r = krao.shape[1]
        if right == 1:
            return ops.gemm(self.T, (1, I), krao, (r, 1), I, r, left)
        return ops.gemm(self.T, (right, 1, I * right, 0), krao, (r, 1, right * r, 0), I, r, right, kb=left)

    def reconstruct_unfolded(self, mode, krao):
        """factors[mode] @ krao^T laid out as the C-order tensor (only for the MU path)."""
        F = self.factors[mode]
        left, I, right = ops._split(list(self.shape), mode)
        r = F.shape[1]
        K = torch.empty(self.shape, dtype=self.T.dtype, device=self.T.device)
        if right == 1:
            # K[l, i] = sum_q krao[l, q] F[i, q]
            ops.gemm(krao, (r, 1), F, (1, r), left, I, r, out=K, ldc=I, sc_b=0)
        else:
            step = 16384
            for l0 in range(0, left, step):
                nb = min(step, left - l0)
                # K[l, i, rr] = sum_q F[i, q] krao[l*right + rr, q]
                ops.gemm(F, (r, 1, 0, 0), krao.reshape(-1)[l0 * right * r:], (1, r, 0, right * r), I, right, r,
                         batch=nb, out=K.reshape(-1)[l0 * I * right:], ldc=right, sc_b=I * right)
        return K

    def step_async(self, rank, norm_tensor, update_rule, beta, sparsity, fixed_modes, normalize):
        """One pass over the modes; returns the device vector of cost terms (no synchronisation).  With direct_cost() the
        terms describe the state the iteration STARTED from (its first pass forms that residual); else the state it ends in."""
        modes = [m for m in range(len(self.shape)) if m not in fixed_modes]
        rhs = krao = cross = None
        mode = None
        direct = self.direct_cost(update_rule, fixed_modes)
        mu_fused = direct and update_rule == "mu"          # MU on the tensor core: no tensor-sized model (_mu_pass)
        lag_terms = res_mode = None
        if direct:
            lag_terms = []
            res_mode = self._mu_cost_mode(beta, fixed_modes) if mu_fused else self._residual_mode(fixed_modes)
            if res_mode not in modes:
                # mode 0 is fixed and the first free mode a view: a pass over unfold(T, 0) just for the residual
                lag_terms.append(self._residual_pass(res_mode)[1])
            for idx, sp in enumerate(sparsity):
                if sp:
                    lag_terms.append(ops.norm1(self.factors[idx]))          # of the incoming state, like the residual
        for mode in modes:
            others = [i for i in range(len(self.factors)) if i != mode]
            fused_krao = update_rule == "hals" and self.plans is not None and len(others) == 2
            krao = None if fused_krao or mu_fused else self.khatri_rao(mode)
            if update_rule == "hals":
                cross = None
                for i in others:
                    gram = self._gram(i)                                     # F_i^T F_i, ntf.py:445
                    cross = gram.clone() if cross is None else ops.hadamard_(cross, gram)
                if mode == res_mode:
                    # first free mode: the fused pass yields the MTTKRP AND the residual of the incoming state
                    rhs_t, res_in = self._residual_pass(mode)
                    lag_terms.insert(0, res_in)
                    rhs = None
                elif fused_krao:
                    # MTTKRP (ntf.py:448-449) on tcgen05: the Khatri-Rao operand goes straight into its bf16 planes
                    self.plans[mode].set_krao(self.factors_t[others[0]], self.factors_t[others[1]])
                    rhs_t = self.plans[mode].cross(0, None)                  # (unfold(T, mode) @ krao)^T
                    rhs = None
                elif self.plans is not None:
                    rhs_t = self.plans[mode].cross(0, ops.transpose(krao))
                    rhs = None
                else:
                    rhs = self.mttkrp(mode, krao)
                    rhs_t = ops.transpose(rhs)
                Ft = self.factors_t[mode].clone()
                nnls.hals_nnls_device(rhs_t, cross, Ft, rank, maxiter=100, delta=0.01,
                                      sparsity_coefficient=sparsity[mode], normalize=normalize[mode],
                                      nonzero=False, result=self.stats)    # ntf.py:454-456
                self.factors_t[mode] = Ft
                self.factors[mode] = ops.transpose(Ft)
                self._gram_ok[mode] = False
            elif mu_fused:
                if beta == 2:
                    # numerator: the MTTKRP (ntf.py:449); denominator: F krao^T krao = F (Hadamard product of the other Grams)
                    cross = None
                    for i in others:
                        gram = self._gram(i)
                        cross = gram.clone() if cross is None else ops.hadamard_(cross, gram)
                    if mode == res_mode:
                        rhs_t, res_in = self._residual_pass(mode)
                        lag_terms.insert(0, res_in)
                    else:
                        self.plans[mode].set_krao(self.factors_t[others[0]], self.factors_t[others[1]])
                        rhs_t = self.plans[mode].cross(0, None)
                    Ft = self.factors_t[mode]
                    Ft = ops.mu_apply(Ft, rhs_t, den_mat=ops.matmul(cross, Ft), floor=mu.epsilon)
                else:
                    cost = self._mu_pass(mode, beta, mode == res_mode)
                    if mode == res_mode:
                        lag_terms.insert(0, cost)
                    Ft = self._mu_finish(mode, beta)
                self.factors_t[mode] = Ft
                self.factors[mode] = ops.transpose(Ft)
                self._gram_ok[mode] = False
            else:
                F = self.factors[mode]
                K = self.reconstruct_unfolded(mode, krao)
                self.factors[mode] = self._mu_factor(F, krao, K, mode, beta)   # ntf.py:459-460
                self.factors_t[mode] = ops.transpose(self.factors[mode])
                self._gram_ok[mode] = False
        if direct:
            return torch.cat([t.reshape(1).to(torch.float64) for t in lag_terms])
        # the cost terms stay on the device: [rec part a, rec part b, sparsity l1 norms...] (see finish_cost)
        terms = []
        F = self.factors[mode]
        if update_rule == "hals":
            # ntf.py:470; ||F krao^T||^2 = <F^T F, krao^T krao> and krao^T krao = cross (Hadamard of Grams)
            ftf = self._gram(mode)
            inner = ops.dot(F, rhs) if rhs is not None else ops.dot(Ft, rhs_t)     # <F, rhs>, either layout
            terms += [inner, ops.dot(ftf, cross)]
        else:
            K = self.reconstruct_unfolded(mode, self.khatri_rao(mode) if krao is None else krao)
            terms += [ops.beta_divergence(self.T, K, beta)]                 # ntf.py:473
        for idx, s in enumerate(sparsity):
            if s:
                terms.append(ops.norm1(self.factors[idx]))                  # ntf.py:463-466
        return torch.cat([t.reshape(1).to(torch.float64) for t in terms])

    @staticmethod
    def finish_cost(terms_host, norm_tensor, update_rule, sparsity, direct=False, beta=2):
        """ntf.py:463-475 from the device terms of step_async (host float64 arithmetic, as in the reference)."""
        if direct:
            # MU, beta = 2: the beta-divergence of ntf.py:473 is half the squared residual
            rec_error = terms_host[0] / 2 if update_rule == "mu" and beta == 2 else terms_host[0]
            rest = terms_host[1:]
        elif update_rule == "hals":
            rec_error = norm_tensor ** 2 - 2 * terms_host[0] + terms_host[1]
            rest = terms_host[2:]
        else:
            rec_error = terms_host[0]
            rest = terms_host[1:]
        sparsity_error = 0.0
        for s, l1 in zip([s for s in sparsity if s], rest):
            sparsity_error += 2 * (s * float(l1))
        return float((rec_error + sparsity_error) / (norm_tensor ** 2))

    def step(self, rank, norm_tensor, update_rule, beta, sparsity, fixed_modes, normalize):
        terms = self.step_async(rank, norm_tensor, update_rule, beta, sparsity, fixed_modes, normalize)
        direct = self.direct_cost(update_rule, fixed_modes)
        if direct:                                      # the terms of the step describe the state it started from
            terms = self.cost_terms_now(sparsity, fixed_modes, update_rule, beta)
        return self.finish_cost(terms.cpu().numpy(), norm_tensor, update_rule, sparsity, direct, beta)

    def _mu_factor(self, F, krao, K, mode, beta):
        """mu_betadivmin(F, krao.T, unfold(T, mode), beta) with the unfolding kept implicit."""
        from nn_fac.utils.beta_divergence import gamma_beta
        left, I, right = ops._split(list(self.shape), mode)
        r = F.shape[1]
        g = gamma_beta(beta)
        if beta == 2:
            P, Q = self.T, K
        elif beta == 1:
            P, Q = ops.mu_terms(K, self.T, beta, want_q=False, out_p=K)[0], None
        else:
            P, Q = ops.mu_terms(K, self.T, beta, want_q=True, out_p=torch.empty_like(K), out_q=K)

        def contract(Z):
            if right == 1:
                return ops.gemm(Z, (1, I), krao, (r, 1), I, r, left)
            return ops.gemm(Z, (right, 1, I * right, 0), krao, (r, 1, right * r, 0), I, r, right, kb=left)

        num = contract(P)
        if Q is None:
            den_vec = ops.row_sums(ops.transpose(krao))                     # column sums of krao = row sums of krao^T
            return ops.mu_apply(F, num, den_vec=den_vec, vec_per_row=False, gamma=g, floor=mu.epsilon)
        return ops.mu_apply(F, num, den_mat=contract(Q), gamma=g, floor=mu.epsilon)


def _pack(factors, like, dtype=None):
    if dtype is not None:
        factors = [f.to(dtype) if f.dtype != dtype else f for f in factors]    # small float32 problems compute in float64 (config.py)
    if isinstance(like, torch.Tensor):
        return factors
    host = [f.cpu().numpy() for f in factors]
    if len({f.shape for f in host}) == 1:
        return np.array(host)                                               # ntf.py:342-344
    out = np.empty(len(host), dtype=object)
    for i, f in enumerate(host):
        out[i] = f
    return out


def compute_ntf(tensor_in, rank, factors_in, n_iter_max=100, tol=1e-8,
                update_rule="hals", beta=2,
                sparsity_coefficients=[], fixed_modes=[], normalize=[],
                verbose=False, return_costs=False):
    """Outer loop of ntf.py:201-344.  The cost is normalised by ||tensor||^2 (ntf.py:475)."""
    nb_modes = len(tensor_in.shape)
    if sparsity_coefficients is None or len(sparsity_coefficients) != nb_modes:      # ntf.py:292-301
        print("Irrelevant number of sparsity coefficient (different from the number of modes), they have been set to None.")
        sparsity_coefficients = [None for _ in range(nb_modes)]
    if fixed_modes is None:
        fixed_modes = []
    if normalize is None or len(normalize) != nb_modes:
        print("Irrelevant number of normalization booleans (different from the number of modes), they have been set to False.")
        normalize = [False for _ in range(nb_modes)]
    _check_step_arguments(update_rule, beta)
    for fixed_value in fixed_modes:
        sparsity_coefficients[fixed_value] = None                           # ntf.py:428-429 (caller's list, as in the reference)
    dt, dt_out = L.working_dtype(int(np.prod(np.shape(tensor_in))), tensor_in, *factors_in)
    state = DeviceNTF(tensor_in, factors_in, dt)
    norm_tensor = float(np.sqrt(ops.sq_diff(state.T).item()))              # ntf.py:290
    cost_fct_vals, toc = [], []
    tic = time.time()
    # The cost of iteration t is read while iteration t+1 is already queued (no idle device between iterations); if the
    # reference's stop test (ntf.py:337) fires on it, the speculative iteration is dropped (factors are replaced, not
    # modified in place, so the previous list is simply kept).
    host = torch.zeros(8, dtype=torch.float64).pin_memory()
    pending = None                                     # (terms on host buffer, event, factors after that iteration)
    # From the second iteration on the outer iteration is one CUDA-graph launch (_graph.py); NNFAC_NTF_GRAPH=0 keeps every
    # iteration eager.
    graphed = None
    use_graph = n_iter_max >= 4 and state.T.is_cuda and os.environ.get("NNFAC_NTF_GRAPH", "1") != "0"
    lagged = state.direct_cost(update_rule, fixed_modes)
    step = lambda: state.step_async(rank, norm_tensor, update_rule, beta, sparsity_coefficients, fixed_modes, normalize)  # noqa: E731

    def record(cost):
        """Append one objective value; returns True when the reference's stop test (ntf.py:337) fires on it."""
        toc.append(time.time() - tic)
        cost_fct_vals.append(cost)
        if verbose:
            if len(cost_fct_vals) == 1:
                print('Normalized cost function value={}'.format(cost))
            else:
                gain = cost_fct_vals[-2] - cost_fct_vals[-1]
                line = 'Normalized cost function value={}, variation={}.'.format(cost_fct_vals[-1], gain)
                print(line if gain > 0 else '\033[91m' + line + '\033[0m')
        if len(cost_fct_vals) >= 2 and abs(cost_fct_vals[-2] - cost_fct_vals[-1]) < tol:
            if verbose:
                print('Converged in {} iterations.'.format(len(cost_fct_vals) - 1))
            return True
        return False

    if lagged:
        # Direct residual (DeviceNTF.direct_cost): round k launches iteration k (state k -> k + 1) -- or, at k = n_iter_max, the
        # closing pass -- and its terms are the objective of state k.  They are read one round later, while the next iteration
        # is already queued, so a stop decision on state s is taken when the device is two iterations ahead: both are dropped.
        hosts = [torch.zeros(8, dtype=torch.float64).pin_memory() for _ in range(2)]
        history = []                                   # eager launches: (factors, factors_t) each iteration started from
        pending, stopped = None, False
        for k in range(n_iter_max + 1):
            if k < n_iter_max:
                if use_graph and k == 1 and graphed is None:
                    graphed = try_capture(state.T.device, state.get_state, state.set_state, step, state.invalidate)
                if graphed is not None:
                    terms = graphed.replay()
                else:
                    history = (history + [(list(state.factors), list(state.factors_t))])[-2:]
                    terms = step()
            else:
                terms = state.cost_terms_now(sparsity_coefficients, fixed_modes, update_rule, beta)
            buf = hosts[k & 1]
            buf[:terms.numel()].copy_(terms, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            entries = [pending] if pending is not None else []
            pending = (ev, buf, terms.numel(), k)
            if k == n_iter_max:
                entries.append(pending)
            for ev_s, buf_s, n_s, s_idx in entries:
                if s_idx == 0:
                    continue                           # objective of the initial factors: the reference never reports it
                ev_s.synchronize()
                cost = state.finish_cost(buf_s[:n_s].numpy().copy(), norm_tensor, update_rule, sparsity_coefficients, True, beta)
                if record(cost) and s_idx < n_iter_max:
                    back = min(k + 1, n_iter_max) - s_idx  # iterations launched beyond state s_idx: 2, or 1 in the closing round
                    if graphed is not None:
                        graphed.roll_back(back)
                    else:
                        state.factors, state.factors_t = history[-back]
                    state.invalidate()
                    stopped = True
                    break
            if stopped:
                break
        out = _pack(state.factors, tensor_in, dt_out)
        if return_costs:
            return out, cost_fct_vals, toc
        return out

    for iteration in range(n_iter_max + 1):
        if iteration < n_iter_max:
            if use_graph and iteration == 1 and graphed is None:
                graphed = try_capture(state.T.device, state.get_state, state.set_state, step, state.invalidate)
            if graphed is not None:
                terms = graphed.replay()
            else:
                before = list(state.factors)
                terms = step()
        if pending is not None:
            ev, nterms, kept = pending
            ev.synchronize()
            cost = state.finish_cost(host[:nterms].numpy().copy(), norm_tensor, update_rule, sparsity_coefficients)
            if record(cost):
                if iteration < n_iter_max:             # drop the speculative iteration
                    if graphed is not None:
                        graphed.roll_back()
                    else:
                        state.factors = before
                        state.factors_t = [ops.transpose(f) for f in before]
                    state.invalidate()
                break
        if iteration == n_iter_max:
            break
        host[:terms.numel()].copy_(terms, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        pending = (ev, terms.numel(), None)
    out = _pack(state.factors, tensor_in, dt_out)
    if return_costs:
        return out, cost_fct_vals, toc
    return out


def one_ntf_step(unfolded_tensors, rank, in_factors, norm_tensor, update_rule, beta,
                 sparsity_coefficients, fixed_modes, normalize,
                 alpha=0.5, delta=0.01):
    """One pass over the modes (ntf.py:347-477).  Takes the reference's list of mode unfoldings;
    only unfolded_tensors[0] (I_0 x prod(others), C order) and the factor shapes are needed to
    rebuild the tensor.  `alpha` is ignored (deterministic rule); `delta` must be 0.01."""
    _check_step_arguments(update_rule, beta)
    for fixed_value in fixed_modes:
        sparsity_coefficients[fixed_value] = None
    shape = tuple(int(f.shape[0]) for f in in_factors)
    first = unfolded_tensors[0]
    tensor = first.reshape(shape) if isinstance(first, torch.Tensor) else np.reshape(first, shape)
    dt = L.resolve_dtype(first, *in_factors)
    state = DeviceNTF(tensor, in_factors, dt)
    cost = state.step(rank, float(norm_tensor), update_rule, beta, sparsity_coefficients, fixed_modes, normalize)
    factors = [L.as_output(f) for f in state.factors]
    factors = factors if isinstance(first, torch.Tensor) else [f.cpu().numpy() for f in factors]
    return factors, cost
