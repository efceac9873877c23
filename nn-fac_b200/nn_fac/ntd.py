"""Nonnegative Tucker decomposition (NTD), B200 path (reference: nn_fac/ntd.py).

``update_rule="mu"`` (any beta >= 0): ``one_ntd_step_mu`` = per-mode ``mu_betadivmin`` on the implicit unfoldings
followed by ``mu_tensorial`` on the core and the beta-divergence cost (ntd.py:658-698).
``update_rule="hals"`` (the reference's default): ``one_ntd_step`` = per-mode HALS solve on the Tucker Grams and a
projected-gradient loop on the core whose stop test runs on the device (ntd.py:436-645), deterministic inner rule.
"""
import os
import time
import warnings

import numpy as np
import torch

import nn_fac.update_rules.mu as mu
import nn_fac.utils.errors as err
import nn_fac.utils.initialize_factors as init_factors
from nn_fac import _lib as L
from nn_fac._graph import try_capture
from nn_fac import _ops as ops
from nn_fac.utils.beta_divergence import gamma_beta


def ntd(tensor, ranks, init="random", core_0=None, factors_0=[], n_iter_max=100, tol=1e-6,
        update_rule="hals", beta=2,
        sparsity_coefficients=[], fixed_modes=[], normalize=[], mode_core_norm=None,
        verbose=False, return_costs=False, deterministic=False, seed=0):
    """Arguments, defaults, checks and returns follow nn_fac.ntd.ntd (ntd.py:27-246):
    returns (core, factors) or (core, factors, cost_fct_vals, toc)."""
    nb_modes = len(tensor.shape)
    if deterministic:
        np.random.seed(seed)                                                # ntd.py:206-207
    if type(ranks) is int:
        ranks = [ranks for _ in range(nb_modes)]
    elif len(ranks) != nb_modes:
        raise err.InvalidRanksException(
            "The number of ranks is different than the dim of the tensor, which is incorrect.") from None
    for i in range(nb_modes):
        if ranks[i] > tensor.shape[i]:                                      # ntd.py:215-219 (mutates the caller's list)
            ranks[i] = tensor.shape[i]
            warnings.warn(f"The {i}-th mode rank was larger than the shape of the tensor, which is incorrect "
                          f"(rank: {ranks[i]}, tensor shape: {tensor.shape[i]}). The rank was then set to the shape of the tensor.")
    if update_rule == "hals":
        assert beta == 2, ("Beta parameter is only used for MU update rule. Please set update_rule to 'mu' to use "
                           f"another beta value than 2. (Current setting: beta = {beta} and update_rule = {update_rule}).")
    if init.lower() == "custom":                                            # ntd.py:224-234
        factors = factors_0
        core = core_0
        if len(factors) != nb_modes:
            raise err.CustomNotEngouhFactors("Custom initialization, but not enough factors")
        for array in factors:
            if array is None:
                raise err.CustomNotValidFactors("Custom initialization, but (at least) one factor is set to 'None'")
        if core is None:
            raise err.CustomNotValidCore("Custom initialization, but the core is set to 'None'")
    else:
        host = tensor.detach().cpu().numpy() if isinstance(tensor, torch.Tensor) else tensor
        core, factors = init_factors.ntd_initialization(host, ranks, init, deterministic=deterministic, seed=seed)
    if init.lower() == "chromas" and 0 not in fixed_modes:
        fixed_modes.append(0)
    return compute_ntd(tensor, ranks, core, factors, n_iter_max=n_iter_max, tol=tol, update_rule=update_rule,
                       beta=beta, sparsity_coefficients=sparsity_coefficients, fixed_modes=fixed_modes,
                       normalize=normalize, mode_core_norm=mode_core_norm, verbose=verbose,
                       return_costs=return_costs, deterministic=deterministic, seed=seed)


class DeviceNTD:
    """Tensor, core and factors resident on one GPU; one call of step_mu = one outer iteration."""

    def __init__(self, tensor, core, factors, dtype, device=None):
        self.T = L.to_device(tensor, dtype, device)
        self.core = L.to_device(core, dtype, device)
        self.factors = [L.to_device(f, dtype, device) for f in factors]
        self.stats = torch.zeros(4, dtype=torch.float64, device=self.T.device)
        # fp32, every rank <= 64: every pass over the tensor runs on tcgen05 over ONE copy of it as bf16 hi/lo planes (4 bytes per
        # element).  The factor update of mode n is the update of U for X = unfold(T, n), V = unfold(G x_{j != n} F_j, n) -- one
        # fused pass (beta = 2: one cross product), model tile and ratios on chip -- on plans[n]: the plan that owns the planes
        # for mode 0, a view of them (NMFPlan.view) for the other modes, or, where an unfolding cannot be addressed in place, a
        # one-sided plan on a copy of it.  core_plan reads the same planes as unfold(T, 0)^T (rows: the columns of unfold(T, 0),
        # contraction over I_0): every contraction of the tensor over mode 0 -- the core update's, HALS's T x_0 F_0^T -- runs
        # there.  Not enough memory for the plans: the strided CUDA-core route (self.plans None), as NNFAC_NTD_TC=0 selects.
        self.plans = self.core_plan = None
        self._m0_ready = False                                              # see step_mu_async
        self._pg, self._pg_calls = None, 0                                  # see _core_loop_graphed
        self._m0_den = torch.empty(int(self.factors[0].shape[1]), dtype=dtype, device=self.T.device)
        self._m0_num = None
        if (dtype == torch.float32 and self.T.dim() >= 2 and max(int(f.shape[1]) for f in self.factors) <= 64
                and os.environ.get("NNFAC_NTD_TC", "1") != "0"):
            try:
                self._build_plans()
            except torch.cuda.OutOfMemoryError:
                self.plans = self.core_plan = None
                torch.cuda.empty_cache()

    def _build_plans(self):
        shape = list(self.T.shape)
        ranks = [int(f.shape[1]) for f in self.factors]
        base = ops.NMFPlan(self.T.reshape(shape[0], -1)).bind_rank(ranks[0], sides=1)
        plans = [base]
        for mode in range(1, len(shape)):
            left, I, right = ops._split(shape, mode)
            view = base.view(left, I, right, ranks[mode])
            if view is None:
                view = ops.NMFPlan(self._unfold(self.T, mode)).bind_rank(ranks[mode], sides=1)
            plans.append(view)
        core = base.view(shape[0], base.n, 1, ranks[0])                    # the last-mode view of (I_0, prod of the others)
        if core is None:
            core = ops.NMFPlan(ops.transpose(self.T.reshape(shape[0], -1))).bind_rank(ranks[0], sides=1)
        self.plans, self.core_plan = plans, core

    def invalidate(self):
        """Core / factors were replaced from outside: nothing left in the plans refers to them."""
        self._m0_ready = False

    def get_state(self):
        return [self.core] + list(self.factors)

    def set_state(self, tensors):
        self.core, self.factors = tensors[0], list(tensors[1:])

    def factor_update(self, mode, beta):
        """mu_betadivmin(F, unfold(G x_{j != mode} F_j, mode), unfold(T, mode), beta), ntd.py:672."""
        F = self.factors[mode]
        B = ops.multi_mode_dot(self.core, self.factors, skip=mode)          # shape of T except R_mode along `mode`
        if self.plans is not None:
            # B_(n) = unfold(B, mode) is installed straight from B: the contraction order of the plan of `mode` (view or copy)
            # is the column order of unfold(T, mode), which is that of unfold(B, mode)
            plan = self.plans[mode]
            left, _, right = ops._split(list(self.T.shape), mode)
            Ft = ops.transpose(F)
            plan.set_operand(B, left, right)
            if beta == 2:
                return self._mu_finish(mode, beta, Ft, plan.cross(0, None))
            plan.set_factor_rows(Ft)
            if beta == 1:
                plan.fused(0, 1, want_cost=False, keep_partials=True)       # (X / (F B_(n))) B_(n)^T, mu.py:82-85
                # row sums of B_(n) (mu.py:86) = G x_{j != n} (column sums of F_j): B_n is not read again
                sums = [None if j == mode else ops.row_sums(ops.transpose(f)).reshape(1, -1) for j, f in enumerate(self.factors)]
                return self._mu_finish(mode, beta, Ft, ops.multi_mode_dot(self.core, sums, skip=mode).reshape(-1))
            plan.fused_beta(0, beta, want_cost=False)
            return self._mu_finish(mode, beta, Ft)
        K = ops.mode_dot(B, F, mode)                                        # = F @ unfold(B, mode), folded (mu.py:82)
        g = gamma_beta(beta)
        if beta == 2:
            P, Q = self.T, K
        elif beta == 1:
            P, Q = ops.mu_terms(K, self.T, beta, want_q=False, out_p=K)[0], None
        else:
            P, Q = ops.mu_terms(K, self.T, beta, want_q=True, out_p=torch.empty_like(K), out_q=K)
        num = ops.unfold_times(P, B, mode)
        if Q is None:
            ones = torch.ones((), dtype=self.T.dtype, device=self.T.device)
            den_vec = ops.unfold_times(ones, B, mode)                       # row sums of unfold(B, mode), mu.py:86
            return ops.mu_apply(F, num, den_vec=den_vec, vec_per_row=False, gamma=g, floor=mu.epsilon)
        return ops.mu_apply(F, num, den_mat=ops.unfold_times(Q, B, mode), gamma=g, floor=mu.epsilon)

    def _mu_finish(self, mode, beta, Ft, extra=None):
        """The update of factor `mode` (given as F^T) from the last pass over its plan, mu.py:84-97: beta = 2, `extra` is the
        numerator B_(n) unfold(T, mode)^T and the denominator (B_(n) B_(n)^T) F^T; beta = 1, `extra` = the row sums of B_(n);
        any other beta, both partial sets of the plan's fused_beta pass."""
        if beta == 2:
            return ops.transpose(ops.mu_apply(Ft, extra, den_mat=ops.matmul(self._bbt(mode), Ft), floor=mu.epsilon))
        if beta == 1:
            return ops.transpose(self.plans[mode].mu_finish_rows(Ft, mu.epsilon, den=extra))
        return ops.transpose(self.plans[mode].mu_finish_rows(Ft, mu.epsilon, gamma=gamma_beta(beta)))

    def _bbt(self, mode):
        """B_(n) B_(n)^T = unfold(G x_{j != n} F_j^T F_j, n) unfold(G, n)^T (r_n x r_n), from the Grams: B_n is never read."""
        grams = [None if j == mode else mu.gram(F) for j, F in enumerate(self.factors)]
        return ops.matmul(self._unfold(ops.multi_mode_dot(self.core, grams, skip=mode), mode), self._unfold(self.core, mode).T)

    # ---- HALS factor updates + projected-gradient core update (ntd.py:436-645) ------------------------------
    @staticmethod
    def _unfold(t, mode):
        return t.movedim(mode, 0).reshape(t.shape[mode], -1).contiguous()

    def _project_all_but(self, mode, P0=None):
        """T x_{j != mode} F_j^T (ntd.py:550); mode None: every mode.  With the tcgen05 plans (fp32, ranks <= 64), for a mode
        other than 0, the first contraction -- the only one that reads the whole tensor -- is T x_0 F_0^T = F_0^T unfold(T, 0),
        one cross product on core_plan (P0 when the caller already has it: it depends on F_0 only); the remaining ones act on a
        tensor r_0 / I_0 times smaller."""
        if self.plans is None or mode == 0:
            return ops.multi_mode_dot(self.T, self.factors, skip=mode, transpose=True)
        P = P0 if P0 is not None else self._project_mode0()
        for d in range(1, self.T.dim()):
            if d != mode:
                P = ops.mode_dot(P, self.factors[d], d, transpose=True)
        return P

    def _project_mode0(self):
        """T x_0 F_0^T on core_plan: r_0 x I_1 x ... """
        P = self.core_plan.cross(0, ops.transpose(self.factors[0]))
        return P.reshape([P.shape[0]] + list(self.T.shape[1:]))

    def step_hals_async(self, norm_tensor, sparsity, fixed_modes, normalize, mode_core_norm, delta=0.01):
        """One outer iteration of one_ntd_step (deterministic inner rule); returns the device vector of cost terms
        [<all_MtX, core>, <core x_n MtM_n, core>, l1 norms of the sparse factors..., l1 norm of the core]."""
        import nn_fac.update_rules.nnls as nnls
        nm = self.T.dim()
        modes = [m for m in range(nm) if m not in fixed_modes]
        temp = elemprod = P0 = None                                          # P0: T x_0 F_0^T for the current F_0 (plans only)
        for mode in modes:
            elemprod = list(self.factors)                                    # ntd.py:534-537
            for i, f in enumerate(self.factors):
                if i != mode:
                    r_i = f.shape[1]
                    elemprod[i] = ops.gemm(f, (1, r_i), f, (r_i, 1), r_i, r_i, f.shape[0])
            core_u = self._unfold(self.core, mode)
            UtU = ops.matmul(self._unfold(ops.multi_mode_dot(self.core, elemprod, skip=mode), mode), core_u.T.contiguous())   # ntd.py:539-544
            if self.plans is not None and mode == 0:
                # ntd.py:555-557 in another association: UtM = B_(0) unfold(T, 0)^T, B_0 = G x_{j>0} F_j, one cross product
                B0 = ops.multi_mode_dot(self.core, self.factors, skip=0)
                UtM = self.plans[0].cross(0, B0.reshape(B0.shape[0], -1))
                temp = None
            else:
                if self.plans is not None and P0 is None:
                    P0 = self._project_mode0()                              # one pass serves every mode >= 1 of the iteration
                temp = self._project_all_but(mode, P0)                                                                        # ntd.py:550
                UtM = ops.matmul(core_u, self._unfold(temp, mode).T.contiguous())                                             # ntd.py:555-557 (transposed)
            Ft = ops.transpose(self.factors[mode])
            nnls.hals_nnls_device(UtM, UtU, Ft, Ft.shape[0], maxiter=100, delta=delta, sparsity_coefficient=sparsity[mode],
                                  normalize=normalize[mode], nonzero=False, result=self.stats)   # ntd.py:571-573
            self.factors[mode] = ops.transpose(Ft)
        last = modes[-1]
        F_last = self.factors[last]
        if temp is not None:
            all_MtX = ops.mode_dot(temp, F_last, last, transpose=True)       # ntd.py:581
        else:
            all_MtX = self._project_all_but(None)                           # the last free mode was mode 0
        all_MtM = list(elemprod)                                             # ntd.py:582-583
        r_l = F_last.shape[1]
        all_MtM[last] = ops.gemm(F_last, (1, r_l), F_last, (r_l, 1), r_l, r_l, F_last.shape[0])
        # step = prod 1 / sigma_max(MtM) rounded to 6 decimals (ntd.py:590-594): control scalar from three tiny Grams
        gradient_step = 1.0
        for MtM in all_MtM:
            gradient_step *= 1.0 / float(np.linalg.svd(MtM.double().cpu().numpy(), compute_uv=False)[0])
        gradient_step = round(gradient_step, 6)
        sparse = 0.0 if sparsity[-1] is None else float(sparsity[-1])       # ntd.py:600-603
        if self._pg_calls >= 1 and os.environ.get("NNFAC_NTD_GRAPH", "1") != "0":
            core, state = self._core_loop_graphed(all_MtX, all_MtM, gradient_step, sparse, delta)
        else:
            core = self.core.clone()
            state = torch.tensor([0.0, 1.0, 1.0, 0.0], dtype=torch.float64, device=core.device)
            fast = ops.core_pg_fast(core)
            MtM_c = [M.contiguous() for M in all_MtM] if fast else None
            Z = torch.empty_like(core) if fast else None
            for it in range(300):                                            # ntd.py:607-617, stop test on the device
                if fast:
                    ops.core_pg_step3(core, all_MtX, MtM_c, Z, gradient_step, sparse, delta, state)
                else:
                    P = ops.multi_mode_dot(core, all_MtM)
                    ops.core_pg_step(core, all_MtX, P, gradient_step, sparse, delta, state)
                if it % self.PG_BATCH == self.PG_BATCH - 1 and float(state[3].item()) != 0.0:
                    break
        self._pg_calls += 1
        self.core_steps = state
        if normalize[-1]:                                                    # ntd.py:619-624
            moved = core.movedim(mode_core_norm, 0).contiguous()
            ops.normalize_rows_(moved.reshape(moved.shape[0], -1))
            core = moved.movedim(0, mode_core_norm).contiguous()
        self.core = core
        if self.plans is not None and nm >= 2 and os.environ.get("NNFAC_NTD_DIRECT", "1") != "0":
            # fp32 with plans: the reconstruction error as the DIRECT residual ||unfold(T, 0) - F_0 unfold(G x_{j>0} F_j, 0)||^2,
            # formed on chip by one fused pass over the (L2-resident) tensor, instead of ntd.py:637's
            # ||T||^2 - 2 <all_MtX, G> + <G x_n MtM_n, G>, whose terms are of the size of ||T||^2: in fp32 that formula keeps
            # ~1e-6 ||T||^2 of noise on a normalised cost of a few 1e-4.  NaN in the second slot marks the direct form.
            B0 = ops.multi_mode_dot(core, self.factors, skip=0)
            self.plans[0].set_factor(0, ops.transpose(self.factors[0]))
            self.plans[0].set_factor(1, self._unfold(B0, 0))
            _, res = self.plans[0].fused(0, 0)
            self._m0_ready = False
            terms = [res, torch.full((1,), float("nan"), dtype=torch.float64, device=core.device)]
        else:
            terms = [ops.dot(all_MtX, core), ops.dot(ops.multi_mode_dot(core, all_MtM), core)]      # ntd.py:637
        for idx, sp in enumerate(sparsity):                                  # ntd.py:627-635
            if sp:
                if idx < nm:
                    terms.append(ops.norm1(self.factors[idx]))
                else:
                    terms.append(ops.row_sums(core.reshape(1, -1)))          # ||core||_1: the core is nonnegative
        return torch.cat([t.reshape(1).to(torch.float64) for t in terms])

    PG_BATCH = 25       # projected-gradient steps between two looks of the host at the `done` flag

    def _core_loop_graphed(self, all_MtX, all_MtM, gradient_step, sparse, delta):
        """The loop of ntd.py:607-617 as replays of ONE CUDA graph of PG_BATCH steps (captured at the second outer
        iteration of this object, replayed by every later one): a step is 3 tiny mode products + 2 kernels on a 32^3 core,
        far below the host's launch rate.  Operands live in fixed buffers; step size and sparsity coefficient travel in
        the device state vector (nnfac_core_pg_step_dev), so nothing call-specific is frozen into the graph but delta."""
        pg = self._pg
        if pg is None or pg["delta"] != delta:
            dev = self.core.device
            pg = {"delta": delta, "core": torch.empty_like(self.core), "MtX": torch.empty_like(all_MtX),
                  "MtM": [torch.empty_like(M) for M in all_MtM],
                  "state": torch.zeros(6, dtype=torch.float64, device=dev), "graph": torch.cuda.CUDAGraph()}
            fast = ops.core_pg_fast(self.core)
            Z = torch.empty_like(self.core)
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(pg["graph"]):
                for _ in range(self.PG_BATCH):
                    if fast:
                        ops.core_pg_step3(pg["core"], pg["MtX"], pg["MtM"], Z, 0.0, 0.0, delta, pg["state"], dev_scalars=True)
                    else:
                        P = ops.multi_mode_dot(pg["core"], pg["MtM"])
                        ops.core_pg_step_dev(pg["core"], pg["MtX"], P, delta, pg["state"])
            pg["Z"] = Z
            self._pg = pg
        pg["core"].copy_(self.core)
        pg["MtX"].copy_(all_MtX)
        for d, s_ in zip(pg["MtM"], all_MtM):
            d.copy_(s_)
        pg["state"].copy_(torch.tensor([0.0, 1.0, 1.0, 0.0, gradient_step, sparse], dtype=torch.float64))
        for _ in range(300 // self.PG_BATCH):
            pg["graph"].replay()
            if float(pg["state"][3].item()) != 0.0:
                break
        return pg["core"].clone(), pg["state"][:4].clone()

    @staticmethod
    def finish_cost_hals(terms_host, norm_tensor, sparsity):
        if np.isnan(terms_host[1]):                     # direct residual (see step_hals_async)
            rec_error = terms_host[0]
        else:
            rec_error = norm_tensor ** 2 - 2 * terms_host[0] + terms_host[1]
        sparsity_error = 0.0
        for sp, l1 in zip([sp for sp in sparsity if sp], terms_host[2:]):
            sparsity_error += 2 * (sp * float(l1))
        return float((rec_error + sparsity_error) / (norm_tensor ** 2))      # ntd.py:638 (normalised)

    def step_mu(self, beta, fixed_modes, normalize, mode_core_norm):
        return float(self.step_mu_async(beta, fixed_modes, normalize, mode_core_norm).item())

    def step_mu_async(self, beta, fixed_modes, normalize, mode_core_norm):
        """One outer iteration; returns the cost as a device scalar (no synchronisation)."""
        for mode in [m for m in range(self.T.dim()) if m not in fixed_modes]:
            if mode == 0 and self._m0_ready:
                # the pass this update needs already ran: it is the cost pass that ended the previous iteration (same core,
                # same factors), which left what the update needs in the plan of mode 0, _m0_den or _m0_num
                self.factors[0] = self._mu_finish(0, beta, ops.transpose(self.factors[0]), self._m0_num if beta == 2 else self._m0_den)
            else:
                self.factors[mode] = self.factor_update(mode, beta)
        self._m0_ready = False
        self.core = mu.mu_tensorial_device(self.core, self.factors, self.T, beta, self.core_plan)   # ntd.py:674
        if normalize[-1]:                                                    # ntd.py:676-681
            moved = self.core.movedim(mode_core_norm, 0).contiguous()
            flat = moved.reshape(moved.shape[0], -1)
            ops.normalize_rows_(flat)
            self.core = moved.movedim(0, mode_core_norm).contiguous()
        if self.plans is None:
            K = ops.multi_mode_dot(self.core, self.factors)
            return ops.beta_divergence(self.T, K, beta)                     # ntd.py:694-696 (not normalised)
        # beta_divergence(T, G x_n F_n, beta) without forming the reconstruction: the cost output of a pass over unfold(T, 0)
        # with U = F_0, V = B_(0) = unfold(G x_{j > 0} F_j, 0) (any mode's unfolding gives the same number; mode 0 is used because
        # the same pass, with the same operands, is the first factor update of the NEXT iteration: what it leaves serves it)
        plan = self.plans[0]
        B = ops.multi_mode_dot(self.core, self.factors, skip=0)
        Vm = B.reshape(B.shape[0], -1)
        keep = 0 not in fixed_modes
        if beta == 2:
            # half the direct residual ||unfold(T, 0) - F_0 B_(0)||^2 of one fused pass, whose cross product B_(0) unfold(T, 0)^T
            # is the next mode-0 numerator
            plan.set_factor(0, ops.transpose(self.factors[0]))
            plan.set_factor(1, Vm)
            if self._m0_num is None:
                self._m0_num = torch.empty((plan.r, plan.m), dtype=torch.float32, device=self.T.device)
            _, res = plan.fused(0, 0, out=self._m0_num)
            self._m0_ready = keep
            return ops.axpby(0.5, res, 0.0, res)                            # ntd.py:694-696 (not normalised)
        if not keep:                                                        # a free mode 0 was installed by its update (mu_finish_rows)
            plan.set_factor_rows(ops.transpose(self.factors[0]))
        plan.set_operand(B, 1, Vm.shape[1])
        if beta == 1:
            _, cost = plan.fused(0, 1, want_cost=True, keep_partials=True)
            if keep:
                ops.row_sums(Vm, out=self._m0_den)
        else:
            cost = plan.fused_beta(0, beta, want_cost=True)
        self._m0_ready = keep
        return cost                                                         # ntd.py:694-696 (not normalised)


def compute_ntd(tensor_in, ranks, core_in, factors_in, n_iter_max=100, tol=1e-6,
                update_rule="hals", beta=2,
                sparsity_coefficients=[], fixed_modes=[], normalize=[], mode_core_norm=None,
                verbose=False, return_costs=False, deterministic=False, seed=0):
    """Outer loop of ntd.py:248-433."""
    nb_modes = len(tensor_in.shape)
    if sparsity_coefficients is None or len(sparsity_coefficients) != nb_modes + 1:   # ntd.py:364-378
        print("Irrelevant number of sparsity coefficient (different from the number of modes + 1 for the core), they have been set to None.")
        sparsity_coefficients = [None for _ in range(nb_modes + 1)]
    if fixed_modes is None:
        fixed_modes = []
    if normalize is None or len(normalize) != nb_modes + 1:
        print("Irrelevant number of normalization booleans (different from the number of modes + 1 for the core), they have been set to False.")
        normalize = [False for _ in range(nb_modes + 1)]
    if normalize[-1] and (mode_core_norm is None or mode_core_norm < 0 or mode_core_norm >= nb_modes):
        print("The core was asked to be normalized, but an invalid mode was specified. Normalization has been set to False.")
        normalize[-1] = False
    if not normalize[-1] and (mode_core_norm is not None and 0 <= mode_core_norm < nb_modes):
        print("The core was asked NOT to be normalized, but mode_core_norm was set to a valid norm. Is this a mistake?")
    if update_rule not in ("hals", "mu"):
        raise err.InvalidArgumentValue(
            f"The update rule provided is not valid. Please choose between 'hals' and 'mu' (Got {update_rule}).")
    if beta < 0:
        raise err.InvalidArgumentValue("Invalid value for beta: negative one.") from None
    dt, dt_out = L.working_dtype(int(np.prod(np.shape(tensor_in))), tensor_in, core_in, *factors_in)
    state = DeviceNTD(tensor_in, core_in, factors_in, dt)
    cost_fct_vals, toc = [], []
    tic = time.time()
    # The cost of iteration t is read while iteration t+1 is already queued; if the stop test (ntd.py:421) fires on it,
    # the speculative iteration is dropped (core and factors are replaced, never modified in place).
    hals = update_rule == "hals"
    norm_tensor = None
    if hals:
        norm_tensor = float(np.sqrt(ops.sq_diff(state.T).item()))           # ntd.py:361
        for fixed_value in fixed_modes:                                      # ntd.py:515-516 (caller's list, as in the reference)
            sparsity_coefficients[fixed_value] = None
    host = torch.zeros(8, dtype=torch.float64).pin_memory()
    pending = None
    nterms = 1
    # MU: from the second iteration on the outer iteration is one CUDA-graph launch (the eager iteration is bound by the
    # host's launch rate, not by the device); NNFAC_NTD_GRAPH=0 keeps every iteration eager
    graphed = None
    use_graph = (not hals) and n_iter_max >= 4 and state.T.is_cuda and os.environ.get("NNFAC_NTD_GRAPH", "1") != "0"
    for iteration in range(n_iter_max + 1):
        if iteration < n_iter_max:
            if use_graph and iteration == 1 and graphed is None:
                graphed = try_capture(state.T.device, state.get_state, state.set_state,
                                      lambda: state.step_mu_async(beta, fixed_modes, normalize, mode_core_norm), state.invalidate)
            if graphed is not None:
                cost_dev = graphed.replay()
            else:
                before = (state.core, list(state.factors))
                if hals:
                    cost_dev = state.step_hals_async(norm_tensor, sparsity_coefficients, fixed_modes, normalize, mode_core_norm)
                else:
                    cost_dev = state.step_mu_async(beta, fixed_modes, normalize, mode_core_norm).reshape(1).to(torch.float64)
        if pending is not None:
            pending.synchronize()
            if hals:
                cost = state.finish_cost_hals(host[:nterms].numpy().copy(), norm_tensor, sparsity_coefficients)
            else:
                cost = float(host[0])
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
                if iteration < n_iter_max:                                   # drop the speculative iteration
                    if graphed is not None:
                        graphed.roll_back()
                    else:
                        state.core, state.factors = before
                    state.invalidate()
                break
        if iteration == n_iter_max:
            break
        nterms = cost_dev.numel()
        host[:nterms].copy_(cost_dev, non_blocking=True)
        pending = torch.cuda.Event()
        pending.record()
    core, factors = state.core, state.factors
    if dt_out != dt:                                    # small float32 problems compute in float64 (nn_fac/config.py)
        core, factors = core.to(dt_out), [f.to(dt_out) for f in factors]
    if not isinstance(tensor_in, torch.Tensor):
        core, factors = core.cpu().numpy(), [f.cpu().numpy() for f in factors]
    if return_costs:
        return core, factors, cost_fct_vals, toc
    return core, factors


def one_ntd_step(tensor, ranks, in_core, in_factors, norm_tensor, sparsity_coefficients, fixed_modes, normalize,
                 mode_core_norm, alpha=0.5, delta=0.01):
    """ntd.py:436-645: HALS on every non-fixed factor, projected gradient on the core; returns (core, factors, cost)
    with the cost normalised by ||tensor||^2.  `alpha` is ignored (deterministic inner rule)."""
    for fixed_value in fixed_modes:                                          # ntd.py:515-516
        sparsity_coefficients[fixed_value] = None
    dt = L.resolve_dtype(tensor, in_core, *in_factors)
    state = DeviceNTD(tensor, in_core, in_factors, dt)
    terms = state.step_hals_async(float(norm_tensor), sparsity_coefficients, fixed_modes, normalize, mode_core_norm, delta)
    cost = state.finish_cost_hals(terms.cpu().numpy(), float(norm_tensor), sparsity_coefficients)
    core, factors = L.as_output(state.core), [L.as_output(f) for f in state.factors]
    if isinstance(tensor, torch.Tensor):
        return core, factors, cost
    return core.cpu().numpy(), [f.cpu().numpy() for f in factors], cost


def one_ntd_step_mu(tensor, ranks, in_core, in_factors, beta, norm_tensor,
                    fixed_modes, normalize, mode_core_norm):
    """ntd.py:658-698: returns (core, factors, cost).  Host arrays are uploaded on every call."""
    if beta < 0:
        raise err.InvalidArgumentValue("Invalid value for beta: negative one.") from None
    dt = L.resolve_dtype(tensor, in_core, *in_factors)
    state = DeviceNTD(tensor, in_core, in_factors, dt)
    cost = state.step_mu(beta, fixed_modes, normalize, mode_core_norm)
    core, factors = L.as_output(state.core), [L.as_output(f) for f in state.factors]
    if isinstance(tensor, torch.Tensor):
        return core, factors, cost
    return core.cpu().numpy(), [f.cpu().numpy() for f in factors], cost


def ntd_mu(*args, **kwargs):
    """Deprecated in the reference as well (ntd.py:649-656)."""
    raise DeprecationWarning("The ntd_mu function is deprecated. Please use the ntd function with update_rule='mu' instead.")
