"""Device operators: torch CUDA tensors in, torch CUDA tensors out, every FLOP in libnnfac_b200.

These are the building blocks the drop-in modules (nmf, ntf, ntd, update_rules.*) are written
with.  torch allocates the buffers; it never computes.
"""
import os

import numpy as np
import torch

from . import _lib as L


def _lib():
    return L.load_library()


def gemm(A, a_str, B, b_str, M, N, K, kb=1, batch=1, out=None, ldc=None, sc_b=0):
    """C[b][i][j] = sum_{q<kb} sum_{k<K} A[b*sa_b + q*sa_q + i*sa_i + k*sa_k] * B[b*sb_b + q*sb_q + k*sb_k + j*sb_j].

    a_str = (sa_i, sa_k, sa_q, sa_b); b_str = (sb_k, sb_j, sb_q, sb_b), in elements.
    """
    if out is None:
        out = torch.empty((batch, M, N) if batch > 1 else (M, N), dtype=A.dtype, device=A.device)
        ldc, sc_b = N, M * N
    sa = tuple(a_str) + (0,) * (4 - len(a_str))
    sb = tuple(b_str) + (0,) * (4 - len(b_str))
    L.check(_lib().nnfac_gemm_strided(L.ctx(A.device), L.code_of(A.dtype), L.ptr(out), ldc, sc_b, L.ptr(A), *sa,
                                      L.ptr(B), *sb, M, N, K, kb, batch, L.stream_ptr()))
    return out


def gram(F, out=None):
    """F (r x len, row-major) -> F F^T (r x r): V V^T (nmf.py:407) / U^T U (nmf.py:432) for rank-major factors."""
    r, length = F.shape
    if out is None:
        out = torch.empty((r, r), dtype=F.dtype, device=F.device)
    L.check(_lib().nnfac_gram(L.ctx(F.device), L.code_of(F.dtype), L.ptr(out), out.stride(0), L.ptr(F), F.stride(0), r,
                              length, L.stream_ptr()))
    return out


def matmul(A, B):
    """Row-major A (M x K) @ B (K x N)."""
    M, K = A.shape
    K2, N = B.shape
    assert K == K2
    return gemm(A, (A.stride(0), A.stride(1)), B, (B.stride(0), B.stride(1)), M, N, K)


def transpose(A):
    rows, cols = A.shape
    out = torch.empty((cols, rows), dtype=A.dtype, device=A.device)
    L.check(_lib().nnfac_transpose(L.ctx(A.device), L.code_of(A.dtype), L.ptr(out), rows, L.ptr(A), A.stride(0),
                                   rows, cols, L.stream_ptr()))
    return out


def hals_nnls(UtM, UtU, V, r, maxiter, delta, sparsity, normalize, nonzero, result=None, no_tc=False):
    """In-place accelerated HALS on V (r x n).  Returns the device double[4] result vector.
    no_tc: never the tensor-core sweep (fp32 CUDA-core sweep instead)."""
    n = UtM.shape[1]
    if result is None:
        result = torch.empty(4, dtype=torch.float64, device=V.device)
    flags = (L.HALS_NORMALIZE if normalize else 0) | (L.HALS_NONZERO if nonzero else 0) | (L.HALS_NO_TC if no_tc else 0)
    L.check(_lib().nnfac_hals_nnls(L.ctx(V.device), L.code_of(V.dtype), L.ptr(UtM), UtM.stride(0), L.ptr(UtU),
                                   UtU.stride(0), L.ptr(V), V.stride(0), r, n, maxiter, float(delta),
                                   float(sparsity), flags, L.ptr(result), L.stream_ptr()))
    return result


def hals_solve(UtM, UtU, V_in, V_out, r, maxiter, delta, sparsity, result=None):
    """V_out (r x n) <- hals_nnls_acc(UtM, UtU, V_in), out of place (fp32; V_in / V_out may be strided views)."""
    n = UtM.shape[1]
    if result is None:
        result = torch.empty(4, dtype=torch.float64, device=V_in.device)
    L.check(_lib().nnfac_hals_solve_f32(L.ctx(V_in.device), L.ptr(UtM), UtM.stride(0), L.ptr(UtU), UtU.stride(0), L.ptr(V_in),
                                        V_in.stride(0), L.ptr(V_out), V_out.stride(0), r, n, int(maxiter), float(delta),
                                        float(sparsity), L.ptr(result), L.stream_ptr()))
    return result


def hals_solve_slabs(slabs, ld, nslabs, slab_stride, r_pad, scratch, UtU, V_in, V_out, r, n, maxiter, delta, sparsity, result=None):
    """hals_solve whose right-hand side is the sum of `nslabs` slabs ([r_pad x ld] each, slab_stride floats apart): split-K
    partials, or the inbox the peers' fused passes pushed their partials into (csrc/hals_sweep.cu)."""
    if result is None:
        result = torch.empty(4, dtype=torch.float64, device=V_in.device)
    L.check(_lib().nnfac_hals_solve_slabs_f32(L.ctx(V_in.device), L.ptr(slabs), int(ld), int(nslabs), int(slab_stride), int(r_pad),
                                              L.ptr(scratch), L.ptr(UtU), UtU.stride(0), L.ptr(V_in), V_in.stride(0), L.ptr(V_out),
                                              V_out.stride(0), r, int(n), int(maxiter), float(delta), float(sparsity), L.ptr(result),
                                              L.stream_ptr()))
    return result


def philox_uniform(rows, cols, row0=0, col0=0, seed=0, stream_id=0, scale=1.0, out=None, accumulate=False, device=None):
    """[rows x cols] float32 block of the synthetic matrix (seed, stream_id): element (i, j) = scale * u(row0 + i, col0 + j)."""
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.float32, device=torch.device("cuda", L.device_index(device)))
    L.check(_lib().nnfac_philox_uniform(L.ctx(out.device), L.ptr(out), out.stride(0), rows, cols, int(row0), int(col0), int(seed),
                                        int(stream_id), float(scale), 1 if accumulate else 0, L.stream_ptr()))
    return out


def mu_terms(K, X, beta, want_q=True, out_p=None, out_q=None):
    """P = K^(beta-2) * X, Q = K^(beta-1).  P may alias K when Q is not wanted."""
    P = out_p if out_p is not None else torch.empty_like(K)
    Q = None
    if want_q:
        Q = out_q if out_q is not None else torch.empty_like(K)
    L.check(_lib().nnfac_mu_terms(L.ctx(K.device), L.code_of(K.dtype), float(beta), L.ptr(K), L.ptr(X), L.ptr(P),
                                  L.ptr(Q), K.numel(), L.stream_ptr()))
    return P, Q


def mu_apply(F, num, den_mat=None, den_vec=None, vec_per_row=False, gamma=1.0, floor=1e-12):
    out = torch.empty_like(F)
    rows = F.shape[0]
    cols = F.numel() // rows
    L.check(_lib().nnfac_mu_apply(L.ctx(F.device), L.code_of(F.dtype), L.ptr(out), L.ptr(F), L.ptr(num),
                                  L.ptr(den_mat), L.ptr(den_vec), 1 if vec_per_row else 0, rows, cols,
                                  float(gamma), float(floor), L.stream_ptr()))
    return out


def _scalar(device):
    return torch.empty(1, dtype=torch.float64, device=device)


def beta_divergence(A, B, beta, out=None):
    out = out if out is not None else _scalar(A.device)
    L.check(_lib().nnfac_beta_divergence(L.ctx(A.device), L.code_of(A.dtype), float(beta), L.ptr(A), L.ptr(B),
                                         A.numel(), L.ptr(out), L.stream_ptr()))
    return out


def sq_diff(A, B=None, out=None):
    out = out if out is not None else _scalar(A.device)
    L.check(_lib().nnfac_sq_diff(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), L.ptr(B), A.numel(), L.ptr(out),
                                 L.stream_ptr()))
    return out


def dot(A, B, out=None):
    out = out if out is not None else _scalar(A.device)
    L.check(_lib().nnfac_dot(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), L.ptr(B), A.numel(), L.ptr(out),
                             L.stream_ptr()))
    return out


def row_sums(A, out=None):
    rows, cols = A.shape
    if out is None:
        out = torch.empty(rows, dtype=A.dtype, device=A.device)
    L.check(_lib().nnfac_row_sums(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), A.stride(0), rows, cols, L.ptr(out),
                                  L.stream_ptr()))
    return out


def norm1(A):
    rows, cols = A.shape
    out = _scalar(A.device)
    L.check(_lib().nnfac_norm1(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), A.stride(0), rows, cols, L.ptr(out),
                               L.stream_ptr()))
    return out


def khatri_rao(A, B):
    I, r = A.shape
    J = B.shape[0]
    out = torch.empty((I * J, r), dtype=A.dtype, device=A.device)
    L.check(_lib().nnfac_khatri_rao(L.ctx(A.device), L.code_of(A.dtype), L.ptr(out), L.ptr(A), I, L.ptr(B), J, r,
                                    L.stream_ptr()))
    return out


def hadamard_(A, B):
    L.check(_lib().nnfac_hadamard(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), L.ptr(A), L.ptr(B), A.numel(),
                                  L.stream_ptr()))
    return A


def axpby(a, X, b, Y):
    """a X + b Y for contiguous tensors of the same shape."""
    out = torch.empty_like(X)
    L.check(_lib().nnfac_axpby(L.ctx(X.device), L.code_of(X.dtype), L.ptr(out), float(a), L.ptr(X), float(b), L.ptr(Y), X.numel(),
                               L.stream_ptr()))
    return out


def normalize_rows_(A):
    rows, cols = A.shape
    L.check(_lib().nnfac_normalize_rows(L.ctx(A.device), L.code_of(A.dtype), L.ptr(A), A.stride(0), rows, cols,
                                        L.stream_ptr()))
    return A


# ---- tensor helpers (C-order N-way tensors, no unfolding copies) ---------------------------------
def core_pg_step(core, MtX, P, step, sparse, delta, state):
    """In-place projected-gradient step on the Tucker core (ntd.py:607-617); `state` = device double[4]."""
    L.check(_lib().nnfac_core_pg_step(L.ctx(core.device), L.code_of(core.dtype), L.ptr(core), L.ptr(MtX), L.ptr(P), core.numel(),
                                      float(step), float(sparse), float(delta), L.ptr(state), L.stream_ptr()))


def core_pg_step_dev(core, MtX, P, delta, state):
    """core_pg_step with the step size and the sparsity coefficient in state[4], state[5] (`state` = device double[6])."""
    L.check(_lib().nnfac_core_pg_step_dev(L.ctx(core.device), L.code_of(core.dtype), L.ptr(core), L.ptr(MtX), L.ptr(P), core.numel(),
                                          float(delta), L.ptr(state), L.stream_ptr()))


def core_pg_step3(core, MtX, MtM, Z, step, sparse, delta, state, dev_scalars=False):
    """Projected-gradient step on a 3-way core with ranks <= 64, product core x_n MtM_n included (ntd.py:607-617)."""
    r0, r1, r2 = core.shape
    assert core.is_contiguous() and MtX.is_contiguous() and all(M.is_contiguous() for M in MtM) and Z.numel() >= core.numel()
    L.check(_lib().nnfac_core_pg_step3(L.ctx(core.device), L.code_of(core.dtype), L.ptr(core), L.ptr(MtX), L.ptr(MtM[0]),
                                       L.ptr(MtM[1]), L.ptr(MtM[2]), r0, r1, r2, L.ptr(Z), float(step), float(sparse),
                                       1 if dev_scalars else 0, float(delta), L.ptr(state), L.stream_ptr()))


def core_pg_fast(core):
    return core.dim() == 3 and max(core.shape) <= 64


def _split(shape, mode):
    left = 1
    for s in shape[:mode]:
        left *= s
    right = 1
    for s in shape[mode + 1:]:
        right *= s
    return left, shape[mode], right


def mode_dot(T, M, mode, transpose=False):
    """fold(M @ unfold(T, mode)) (tensorly.tenalg.mode_dot); with transpose=True uses M^T."""
    shape = list(T.shape)
    left, I, right = _split(shape, mode)
    if transpose:
        R, si, sk = M.shape[1], M.stride(1), M.stride(0)
    else:
        R, si, sk = M.shape[0], M.stride(0), M.stride(1)
    shape[mode] = R
    out = torch.empty(shape, dtype=T.dtype, device=T.device)
    if right == 1:
        # out[l, a] = sum_i T[l, i] M[a, i]
        gemm(T, (I, 1), M, (sk, si), left, R, I, out=out, ldc=R, sc_b=0)
    else:
        # out[l, a, rr] = sum_i M[a, i] T[l, i, rr], batched over l (chunked to respect the grid limit)
        step = 16384
        for l0 in range(0, left, step):
            nb = min(step, left - l0)
            gemm(M, (si, sk, 0, 0), T.reshape(-1)[l0 * I * right:], (right, 1, 0, I * right), R, right, I,
                 batch=nb, out=out.reshape(-1)[l0 * R * right:], ldc=right, sc_b=R * right)
    return out


def multi_mode_dot(T, mats, skip=None, transpose=False):
    out = T
    for mode, M in enumerate(mats):
        if mode == skip:
            continue
        out = mode_dot(out, M, mode, transpose=transpose)
    return out


def unfold_times(P, B, mode):
    """unfold(P, mode) @ unfold(B, mode)^T for tensors that differ only along `mode`
    (P: I along mode, B: R along mode).  Result I x R.  P may be a 0-d 'ones' marker (shape ())."""
    shape = list(B.shape)
    left, R, right = _split(shape, mode)
    if P.dim() == 0:
        # ones^T @ unfold(B, mode)^T : row sums of the unfolding
        if right == 1:
            return gemm(P.reshape(1), (0, 0, 0, 0), B, (R, 1, 0, 0), 1, R, left).reshape(R)
        return gemm(P.reshape(1), (0, 0, 0, 0), B, (1, right, R * right, 0), 1, R, right, kb=left).reshape(R)
    I = P.shape[mode]
    if right == 1:
        return gemm(P, (1, I, 0, 0), B, (R, 1, 0, 0), I, R, left)
    return gemm(P, (right, 1, I * right, 0), B, (1, right, R * right, 0), I, R, right, kb=left)


class NMFPlan:
    """Owner of an nnfac_nmf_plan (X resident as bf16 hi/lo planes -- or hi/mid/lo, planes=3 -- in both orientations;
    tcgen05 path)."""

    SLAB_BYTES = 64 << 20     # upload granularity of a host-resident X

    def __init__(self, X, device=None):
        """X: float32 CUDA tensor (m x n), or a host array / CPU tensor, which is uploaded slab by slab with the
        upload of slab i+1 overlapping the ingest of slab i (the fp32 X never exists on the device as a whole)."""
        import ctypes
        if isinstance(X, torch.Tensor) and X.is_cuda:
            assert X.dtype == torch.float32 and X.dim() == 2
            self.device = X.device
        else:
            if not isinstance(X, torch.Tensor):
                X = torch.from_numpy(np.ascontiguousarray(np.asarray(X)))
            assert X.dim() == 2
            X = X.contiguous()
            self.device = torch.device("cuda", L.device_index(device))
        self.m, self.n = X.shape
        self.handle = ctypes.c_void_p()
        self.r = None
        self.planes = 2
        self._xf32 = None
        self._xf32_refused = False
        self._den = None
        self._X = X

    def bind_rank(self, r, sides=3, planes=2):
        """sides: 3 = planes of X and of X^T; 1 = only X (passes over side 0, e.g. the MTTKRP of an unfolding); 2 = only X^T.
        planes: bf16 planes per value, 2 (hi + lo) or 3 (hi + mid + lo, the fp32 values exactly; rank <= 64)."""
        import ctypes
        self.r = r
        self.sides = sides
        self.planes = planes
        # the plan lives in one block of torch's caching allocator: a second factorisation of same-shaped data
        # reuses it without any cudaMalloc / cudaFree
        nbytes = ctypes.c_size_t()
        L.check(_lib().nnfac_nmf_plan_bytes_planes(L.ctx(self.device), self.m, self.n, r, sides, planes, ctypes.byref(nbytes)))
        self._workspace = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        L.check(_lib().nnfac_nmf_plan_create_planes(L.ctx(self.device), self.m, self.n, r, sides, planes, L.ptr(self._workspace),
                                                    nbytes.value, L.stream_ptr(), ctypes.byref(self.handle)))
        if self._X.is_cuda:
            L.check(_lib().nnfac_nmf_plan_load_x(self.handle, L.ptr(self._X), self._X.stride(0), L.stream_ptr()))
        else:
            self._load_host(self._X)
        self._X = None
        return self

    def view(self, left, I, right, r):
        """The I x (left * right) unfolding of the middle axis of the C-order tensor (left, I, right) whose mode-0 unfolding this
        plan holds, addressed in place (nnfac_nmf_plan_create_view).  Returns None when the extents do not allow it."""
        import ctypes
        nbytes = ctypes.c_size_t()
        rc = _lib().nnfac_nmf_plan_view_bytes(L.ctx(self.device), self.handle, left, I, right, r, ctypes.byref(nbytes))
        if rc == L.ERR_UNSUPPORTED:
            return None
        L.check(rc)
        v = NMFPlan.__new__(NMFPlan)
        v.device, v.m, v.n, v.r, v.sides, v.planes = self.device, I, left * right, r, 1, 2
        v._xf32, v._xf32_refused, v._X, v._base = None, True, None, self          # keeps the base plan (and its planes) alive
        v._den = None
        v._workspace = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        v.handle = ctypes.c_void_p()
        L.check(_lib().nnfac_nmf_plan_create_view(L.ctx(self.device), self.handle, left, I, right, r, L.ptr(v._workspace), nbytes.value,
                                                  L.stream_ptr(), ctypes.byref(v.handle)))
        return v

    def _load_host(self, host):
        """Double-buffered upload + ingest: copy stream fills slab b while the main stream splits slab 1-b into planes."""
        m, n = self.m, self.n
        rows_per = max(32, (self.SLAB_BYTES // max(1, n * host.element_size())) // 32 * 32)
        rows_per = min(rows_per, m)
        main = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(main)
        bufs = [torch.empty((rows_per, n), dtype=host.dtype, device=self.device) for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        ingested = [torch.cuda.Event() for _ in range(2)]
        for i, r0 in enumerate(range(0, m, rows_per)):
            b, rows = i & 1, min(rows_per, m - r0)
            with torch.cuda.stream(side):
                if i >= 2:
                    side.wait_event(ingested[b])
                bufs[b][:rows].copy_(host[r0:r0 + rows], non_blocking=True)
                copied[b].record(side)
            main.wait_event(copied[b])
            slab = bufs[b][:rows]
            if slab.dtype != torch.float32:
                slab = slab.float()
            L.check(_lib().nnfac_nmf_plan_load_x_rows(self.handle, L.ptr(slab), slab.stride(0), r0, rows, L.stream_ptr()))
            ingested[b].record(main)
        L.check(_lib().nnfac_nmf_plan_load_x_done(self.handle, L.stream_ptr()))

    def reduce(self, side, out=None):
        """Sum of the split-K partials the last pass over `side` left in the plan (r x rows of that side)."""
        R = self.m if side == 0 else self.n
        if out is None:
            out = torch.empty((self.r, R), dtype=torch.float32, device=self.device)
        L.check(_lib().nnfac_nmf_plan_reduce(self.handle, side, L.ptr(out), out.stride(0), L.stream_ptr()))
        return out

    def reduce_chunked(self, side, slabs, chunk, tail=None):
        """The sum of reduce(side) as the send buffer of a reduce-scatter over `slabs` ranks: [slabs][r][chunk + t] with the small
        matrix `tail` (r x t) copied behind every chunk."""
        t = 0 if tail is None else int(tail.shape[1])
        out = torch.empty((slabs, self.r, chunk + t), dtype=torch.float32, device=self.device)
        L.check(_lib().nnfac_nmf_plan_reduce_chunked(self.handle, side, L.ptr(out), chunk, slabs, L.ptr(tail),
                                                     tail.stride(0) if tail is not None else 0, t, L.stream_ptr()))
        return out

    def cross(self, which, F, out=None, keep_partials=False):
        """which=0: F = V (r x n) -> V X^T (r x m); which=1: F = U^T (r x m) -> U^T X (r x n).
        F=None: the factor installed with set_factor / mu_finish (its operand planes are reused)."""
        R = self.m if which == 0 else self.n
        if out is None and not keep_partials:
            out = torch.empty((self.r, R), dtype=torch.float32, device=self.device)
        L.check(_lib().nnfac_nmf_plan_cross(self.handle, which, L.ptr(F), F.stride(0) if F is not None else 0, L.ptr(out),
                                            out.stride(0) if out is not None else 0,
                                            L.stream_ptr()))
        return out

    def set_factor(self, which, Ft):
        """which=0: U given as U^T (r x m); which=1: V (r x n).  Rebuilds that factor's bf16 operand planes."""
        L.check(_lib().nnfac_nmf_plan_set_factor(self.handle, which, L.ptr(Ft), Ft.stride(0), L.stream_ptr()))

    def set_factor_gathered(self, which, gathered, length):
        """gathered: [slices][r][chunk] (all-gather of column slices of the factor).  Installs the factor and returns it
        rank-major (r x length)."""
        slices, r, chunk = gathered.shape
        out = torch.empty((r, length), dtype=torch.float32, device=self.device)
        L.check(_lib().nnfac_nmf_plan_set_factor_gathered(self.handle, which, L.ptr(gathered), chunk, L.ptr(out), out.stride(0),
                                                          L.stream_ptr()))
        return out

    def set_krao(self, At, Bt):
        """The r x (I*J) Khatri-Rao factor of two rank-major factors (r x I, r x J) as the operand of cross(0, None)."""
        L.check(_lib().nnfac_nmf_plan_set_krao(self.handle, L.ptr(At), At.stride(0), At.shape[1], L.ptr(Bt), Bt.stride(0),
                                               Bt.shape[1], L.stream_ptr()))

    def set_krao_rows(self, At, Bt):
        """The same Khatri-Rao factor as rank-contiguous planes, the operand of fused(0, 0) (MTTKRP + direct residual)."""
        L.check(_lib().nnfac_nmf_plan_set_krao_rows(self.handle, L.ptr(At), At.stride(0), At.shape[1], L.ptr(Bt), Bt.stride(0),
                                                    Bt.shape[1], L.stream_ptr()))

    def hals_solve(self, which, UtM, UtU, F, maxiter, delta, sparsity, result):
        """hals_nnls_acc(UtM, UtU, F) on the tensor-core sweep with the result installed in the plan by the same kernel.
        Returns the new factor (r x len), or None when the shape is outside that kernel (caller: hals_nnls + set_factor)."""
        out = torch.empty_like(F)
        rc = _lib().nnfac_nmf_plan_hals_solve(self.handle, which, L.ptr(UtM), UtM.stride(0) if UtM is not None else 0, L.ptr(UtU),
                                              UtU.stride(0), L.ptr(F),
                                              F.stride(0), L.ptr(out), out.stride(0), int(maxiter), float(delta), float(sparsity),
                                              L.ptr(result), L.stream_ptr())
        if rc == L.ERR_UNSUPPORTED:
            return None
        L.check(rc)
        return out

    def mu_finish(self, which, F, den, floor):
        """max(F * num / den[:, None], floor) from the numerator partials of the last fused(which, 1, keep_partials=True);
        the result is installed as factor `which` (mu.py:84-88 + set_factor in one kernel)."""
        out = torch.empty_like(F)
        L.check(_lib().nnfac_nmf_plan_mu_finish(self.handle, which, L.ptr(F), F.stride(0), L.ptr(den), float(floor),
                                                L.ptr(out), out.stride(0), L.stream_ptr()))
        return out

    def fused(self, side, mode, want_cost=True, out=None, cost_out=None, keep_partials=False):
        """One fused X pass with the installed factors (rank <= 64).  mode 0: HALS cross product + ||X-UV||^2;
        mode 1: beta=1 MU numerator + KL(X|UV).  Returns (out r x rows, cost device scalar or None).
        keep_partials: leave the split partials in the plan for mu_finish instead of reducing them into `out`."""
        R = self.m if side == 0 else self.n
        if mode == 1:
            self._want_f32()
        if out is None and not keep_partials:
            out = torch.empty((self.r, R), dtype=torch.float32, device=self.device)
        if cost_out is None and (want_cost or mode == 0):
            cost_out = torch.empty(1, dtype=torch.float64, device=self.device)
        L.check(_lib().nnfac_nmf_plan_fused(self.handle, side, mode, 1 if want_cost else 0, L.ptr(out),
                                            out.stride(0) if out is not None else 0, L.ptr(cost_out), L.stream_ptr()))
        return out, cost_out

    def _want_f32(self):
        """The beta = 1 and general-beta passes only need x in registers (never as a tensor-core operand): from an fp32 copy of X
        they save three instructions per element (no bf16 unpack + add).  With the issuing warps converged the beta = 1 pass is
        bound by the issue slots of its transform warps, and the copy pays: MU 905 -> 950 it/s at C2.  It costs 2 x 4mn bytes, so
        it is made on first use only when that leaves at least as much memory free again (NNFAC_MU_F32=0 / 1 force it off / on).
        A 3-plane plan's beta = 1 pass always reads the copy (then the caller's fp32 values)."""
        if self._xf32 is None and self.fused_ok and self.sides == 3 and not self._xf32_refused:
            want = os.environ.get("NNFAC_MU_F32", "auto")
            need = 2 * 4 * self.m * self.n
            if self.planes == 3 or want == "1" or (want != "0" and torch.cuda.mem_get_info(self.device)[0] > 2 * need + (1 << 30)):
                self.enable_f32()
            else:
                self._xf32_refused = True

    def fused_beta(self, side, beta, want_cost=True, cost_out=None):
        """One general-beta pass (beta >= 0 other than 1 and 2, rank <= 64, two planes): the split partials of the numerator
        (K^(beta-2) * X) V^T (side 0; its twin for V on side 1) stay in the plan, those of the denominator K^(beta-1) V^T in a
        buffer the plan object owns; both are consumed by mu_finish_beta.  Returns the cost (device scalar) or None."""
        import ctypes
        self._want_f32()
        if self._den is None:
            nbytes = ctypes.c_size_t()
            L.check(_lib().nnfac_nmf_plan_fused_beta_bytes(self.handle, ctypes.byref(nbytes)))
            self._den = torch.empty(nbytes.value // 4, dtype=torch.float32, device=self.device)
        if cost_out is None and want_cost:
            cost_out = torch.empty(1, dtype=torch.float64, device=self.device)
        L.check(_lib().nnfac_nmf_plan_fused_beta(self.handle, side, float(beta), 1 if want_cost else 0, L.ptr(self._den),
                                                 L.ptr(cost_out), L.stream_ptr()))
        return cost_out

    def mu_finish_beta(self, which, F, gamma, floor):
        """max(F * (num / den)^gamma, floor) from the two partial sets of the last fused_beta(which); the result is installed as
        factor `which` (mu.py:84-97 + set_factor in one kernel)."""
        out = torch.empty_like(F)
        L.check(_lib().nnfac_nmf_plan_mu_finish_beta(self.handle, which, L.ptr(F), F.stride(0), L.ptr(self._den), float(gamma),
                                                     float(floor), L.ptr(out), out.stride(0), L.stream_ptr()))
        return out

    def enable_f32(self):
        """fp32 copies of X / X^T for the beta = 1 fused pass (made from the planes on first use)."""
        import ctypes
        nbytes = ctypes.c_size_t()
        L.check(_lib().nnfac_nmf_plan_f32_bytes(self.handle, ctypes.byref(nbytes)))
        self._xf32 = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        L.check(_lib().nnfac_nmf_plan_enable_f32(self.handle, L.ptr(self._xf32), nbytes.value, L.stream_ptr()))

    @property
    def fused_ok(self):
        """The beta = 1 fused pass (and its fp32 copies of X) cover rank <= 64; the residual pass covers rank <= 128."""
        return self.r is not None and self.r <= 64

    def info(self, which):
        import ctypes
        vals = [ctypes.c_int() for _ in range(5)]
        L.check(_lib().nnfac_nmf_plan_info(self.handle, which, *[ctypes.byref(v) for v in vals]))
        return dict(zip(("splits", "stages_per_unit", "num_units", "num_stages", "grid"), [v.value for v in vals]))

    def __del__(self):
        try:
            if self.handle:
                _lib().nnfac_nmf_plan_destroy(self.handle)      # host bookkeeping only: the workspace is a torch tensor,
                self.handle = None                              # released stream-ordered by the caching allocator
        except Exception:
            pass
