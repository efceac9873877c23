"""fp32 headline path for NMF (rank <= 64): two X passes per outer iteration, everything on tcgen05.

Layout on the device: both factors are kept "rank-major" -- U as U^T (r x m) and V (r x n) -- which is
what the HALS sweep and the GEMM epilogues produce and consume; X lives only as bf16 hi/lo planes in
both orientations (the fp32 upload is dropped after the ingest).

Cost with a lag of one pass: the cost of iteration t needs U_t V_t, which is exactly the model tile
the first pass of iteration t+1 forms (nmf.py:452/455 re-form it in a third pass).  The loop below
therefore learns cost[t] while iteration t+1 is already in flight; if the reference's stop test
(|cost[t-1] - cost[t]| < tol, nmf.py:320) fires, the speculative iteration is discarded.  A final
cost-only pass closes the last iteration.

Several GPUs (one process each): X is sharded by COLUMNS.  Rank p holds X_p (m x n_p) and V_p (r x n_p);
U is replicated.  Per outer iteration there is one exchange step on each side of the U update:
  * the partial cross products of the first pass (V_p X_p^T, r x m) and the partial Gram V_p V_p^T (HALS), or the partial
    MU numerator and the partial row sums of V (MU), are summed, every rank receiving only the rows of U it updates: the
    fused pass of every rank writes its partials straight into the owners' inboxes in peer-mapped memory (PeerExchange);
  * the U update is split by rows of U (columns of U^T): every rank solves / updates its own m/P slice and the install
    kernel reads all slices from their owners' send buffers, so the solve shrinks with P instead of being repeated on every
    rank.  Without peer access the same steps run as NCCL collectives (reduce-scatter / all-reduce, all-gather).
The V side needs no exchange of factor data.  The HALS stop test (nnls.py:156) sums the squared steps over ALL columns
of a solve, also when they are spread over several GPUs: the sweep kernels of all ranks exchange their partial sums once per
sweep through peer-mapped "boards" (8-byte stores over NVLink, csrc/tc_sweep.cu), so a sharded solve stops after exactly
the sweeps of the unsharded one.  (Solves outside the tensor-core sweep -- normalize, slices too wide for tensor memory --
fall back to the CUDA-core kernel with the rule applied per slice.)  Costs are summed with a scalar all-reduce.
"""
import contextlib
import ctypes
import os
import time

import torch

import nn_fac.update_rules.mu as mu
from nn_fac import _lib as L
from nn_fac import _ops as ops
from nn_fac.utils.beta_divergence import gamma_beta

MODE_RES, MODE_MU = 0, 1


def eligible(dtype, rank, update_rule, beta, planes=2):
    """fp32 on the tcgen05 path: HALS and Frobenius MU up to rank 128 (residual + cross-product pass), MU with any other
    beta >= 0 up to rank 64 (beta = 1: one contraction; every other beta: numerator and denominator contractions).
    planes = 3 (precision "fp32x3"): HALS and MU with beta = 1 or 2, up to rank 64."""
    if dtype != torch.float32:
        return False
    if update_rule == "hals" or (update_rule == "mu" and beta == 2):
        return rank <= (128 if planes == 2 else 64)
    if update_rule != "mu" or rank > 64:
        return False
    return beta == 1 or (planes == 2 and beta >= 0)


def general_beta(update_rule, beta):
    """MU with a beta that needs both contractions (the general-beta pass).  FusedNMF.run takes beta = None as 1."""
    return update_rule == "mu" and beta is not None and beta != 1 and beta != 2


def planes_of_precision():
    """bf16 planes per value of the tensor-core NMF path under the current config.precision."""
    from nn_fac import config
    return 3 if config.precision == "fp32x3" else 2


# HALS solves of a 3-plane factorisation run on a copy (the tensor-core sweep inside nnfac_nmf_plan_hals_solve writes two planes)
# through nnfac_hals_nnls, with NNFAC_HALS_NO_TC: the fp32 CUDA-core sweep solves instead of the tensor-core one, whose step
# operand is a bf16 hi/lo split.  At 4096 x 4096, rank 32, near-exact data the tensor-core sweep left the objective 1.6e-4
# away from float64, the CUDA-core sweep 6.7e-5 (DESIGN.md section 1).
TC_SWEEP_FP32X3 = False


# Peer-mapped resources are expensive to set up (cudaMalloc + CUDA IPC export / open on every rank + a barrier: tens of
# milliseconds on 8 GPUs) and independent of the data, so they are kept for the life of the process and shared by every
# factorisation of the same group and shape: boards per (group, device), exchange regions per (group, device, r, m, chunk, tail).
_BOARDS = {}
_EXCHANGES = {}


def release_exchanges():
    """Free the cached exchange regions (every rank of the group must call it at the same point)."""
    for px in list(_EXCHANGES.values()):
        px.close()
    _EXCHANGES.clear()


import atexit  # noqa: E402
atexit.register(release_exchanges)


class Comm:
    """The exchange steps of the column-sharded path over a torch.distributed group (NCCL on GPUs).
    With a single rank every call returns its argument untouched and no collective is issued."""

    def __init__(self, group=None, align=128):
        self.group = group
        self.align = align      # slices of the U solve start on multiples of this many rows of U
        if group is None:
            self.world, self.rank = 1, 0
        else:
            import torch.distributed as dist
            self.dist = dist
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)

    def sum_(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t

    def max_(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t

    def slice_of(self, length):
        """Equal aligned chunks of range(length): returns (chunk, lo, hi) of this rank."""
        chunk = -(-length // self.world)
        chunk = -(-chunk // self.align) * self.align
        lo = min(self.rank * chunk, length)
        return chunk, lo, min(lo + chunk, length)

    def slice_lengths(self, length):
        """Columns of every rank's slice of range(length) (see slice_of)."""
        chunk = -(-length // self.world)
        chunk = -(-chunk // self.align) * self.align
        return [max(0, min((p + 1) * chunk, length) - min(p * chunk, length)) for p in range(self.world)]

    def all_lengths(self, n_local, device):
        """The local column counts of all ranks (the V blocks need not be equal)."""
        if self.world == 1:
            return [int(n_local)]
        t = torch.zeros(self.world, dtype=torch.int64, device=device)
        t[self.rank] = int(n_local)
        self.sum_(t)
        return [int(v) for v in t.cpu().tolist()]

    # ---- the cross-GPU stop scalar of collective HALS solves (GPU ranks only) ----
    _boards_device = None

    def attach_boards(self, device):
        """Once per (group, device): every rank exports the CUDA IPC handle of its board, the handles are all-gathered and
        every rank maps the boards of its peers (nnfac_ctx_board_export / _attach)."""
        if self.world == 1 or self._boards_device == device:
            return self._boards_device is not None
        if self.world > 8:
            return False
        key = (self.group, L.device_index(device))
        if key in _BOARDS:                            # attached by an earlier factorisation over this group
            if _BOARDS[key]:
                self._boards_device = device
            return _BOARDS[key]
        lib = L.load_library()
        mine = (ctypes.c_ubyte * 64)()
        L.check(lib.nnfac_ctx_board_export(L.ctx(device), mine))
        send = torch.tensor(list(mine), dtype=torch.uint8, device=device)
        recv = torch.empty(self.world * 64, dtype=torch.uint8, device=device)
        self.dist.all_gather_into_tensor(recv, send, group=self.group)
        handles = (ctypes.c_ubyte * (64 * self.world))(*recv.cpu().tolist())
        rc = lib.nnfac_ctx_board_attach(L.ctx(device), self.world, self.rank, handles)
        ok = torch.tensor([1 if rc == 0 else 0], dtype=torch.int64, device=device)
        self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN, group=self.group)      # all ranks or none
        _BOARDS[key] = int(ok.item()) == 1
        if _BOARDS[key]:
            self._boards_device = device
            return True
        import warnings
        warnings.warn("nn_fac: peer access between the GPUs of this group is not available (%s); the sharded HALS solves "
                      "apply the stop rule per slice" % L.load_library().nnfac_last_error().decode())
        return False

    @contextlib.contextmanager
    def collective(self, lengths):
        """The tensor-core HALS solves issued inside are one slice each of a joint solve over the group: `lengths` = columns of
        every rank's slice.  No-op for a single rank or without attached boards."""
        if self.world == 1 or self._boards_device is None:
            yield
            return
        lib = L.load_library()
        arr = (ctypes.c_int64 * self.world)(*[int(v) for v in lengths])
        L.check(lib.nnfac_ctx_collective(L.ctx(self._boards_device), 1, arr))
        try:
            yield
        finally:
            L.check(lib.nnfac_ctx_collective(L.ctx(self._boards_device), 0, None))

    def reduce_scatter_columns(self, M, tail, chunk):
        """Sum over the ranks of M (r x length) and of `tail` (r x t), of which this rank only receives its own column slice
        [rank*chunk, (rank+1)*chunk) of M (zero-padded) plus the whole summed tail: one reduce-scatter instead of an
        all-reduce (half the bytes on the wire).  Returns (slice r x chunk, tail r x t)."""
        r, length = M.shape
        t = tail.shape[1]
        if length == self.world * chunk:
            send = torch.empty((self.world, r, chunk + t), dtype=M.dtype, device=M.device)
            send[:, :, :chunk].copy_(M.view(r, self.world, chunk).permute(1, 0, 2))       # one strided copy
        else:
            send = torch.zeros((self.world, r, chunk + t), dtype=M.dtype, device=M.device)
            for p in range(self.world):
                lo, hi = min(p * chunk, length), min((p + 1) * chunk, length)
                if hi > lo:
                    send[p, :, :hi - lo].copy_(M[:, lo:hi])
        send[:, :, chunk:].copy_(tail.unsqueeze(0).expand(self.world, r, t))
        recv = torch.empty((r, chunk + t), dtype=M.dtype, device=M.device)
        self.dist.reduce_scatter_tensor(recv, send.view(self.world * r, chunk + t), op=self.dist.ReduceOp.SUM, group=self.group)
        return recv[:, :chunk], recv[:, chunk:]

    def reduce_scatter_send(self, send):
        """send: [world][r][w] (slab p = what rank p is to receive).  Returns the (r x w) sum over the ranks of this rank's slab."""
        world, r, w = send.shape
        recv = torch.empty((r, w), dtype=send.dtype, device=send.device)
        self.dist.reduce_scatter_tensor(recv, send.view(world * r, w), op=self.dist.ReduceOp.SUM, group=self.group)
        return recv

    def gather_slices(self, send):
        """send: this rank's slice (r x chunk, zero-padded).  Returns [world][r][chunk] (all-gather, no staging copies)."""
        r, chunk = send.shape
        recv = torch.empty((self.world, r, chunk), dtype=send.dtype, device=send.device)
        self.dist.all_gather_into_tensor(recv.view(self.world * r, chunk), send, group=self.group)
        return recv

    def gather_columns_(self, Ft, chunk, lo, hi):
        """Every rank owns columns [lo, hi) of Ft (r x length); afterwards every rank holds all of them."""
        if self.world == 1:
            return Ft
        r, length = Ft.shape
        send = torch.zeros((r, chunk), dtype=Ft.dtype, device=Ft.device)
        send[:, :hi - lo].copy_(Ft[:, lo:hi])
        recv = torch.empty((self.world * r, chunk), dtype=Ft.dtype, device=Ft.device)
        self.dist.all_gather_into_tensor(recv, send, group=self.group)
        Ft.copy_(recv.view(self.world, r, chunk).permute(1, 0, 2).reshape(r, self.world * chunk)[:, :length])
        return Ft


class _RawView:
    """A device pointer owned by libnnfac_b200 as something torch.as_tensor can alias (CUDA array interface v2)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False), "version": 2,
                                         "strides": None}


class PeerExchange:
    """The U-side exchange of the sharded path over peer-mapped memory instead of NCCL (csrc/peer_xchg.cu).  Every rank's stage
    buffer is [tail block r x tpad | inbox (world * splits) x r_pad x chunk]: the peers' fused passes write their partials of this
    rank's rows of U straight into the inbox (nnfac_nmf_plan_set_push), the first t columns of the tail block carry this rank's
    partial Gram or row sums.  The slice results go to the send buffers [r x (chunk + tpad)] (the slice's Gram behind the slice),
    and the install kernel reads all slices from the peers' send buffers.  One region per FusedNMF state."""

    def __init__(self, comm, device, r, chunk, tail, splits):
        """splits: split-K partials per row tile of the fused pass over side 0 (the inbox holds world * splits slabs)."""
        lib = L.load_library()
        self.comm, self.device, self.r, self.chunk, self.tail = comm, device, r, chunk, tail
        self.tpad = -(-tail // 4) * 4                 # row pitches stay multiples of 4 floats: 16-byte loads over NVLink
        self.r_pad = -(-r // 16) * 16
        self.nslabs, self.slab_stride = comm.world * splits, self.r_pad * chunk
        self.inbox_off = r * self.tpad
        self.handle = ctypes.c_void_p()
        L.check(lib.nnfac_xchg_create(L.ctx(device), self.inbox_off + self.nslabs * self.slab_stride, r * (chunk + self.tpad),
                                      ctypes.byref(self.handle)))
        mine = (ctypes.c_ubyte * 64)()
        L.check(lib.nnfac_xchg_export(self.handle, mine))
        send = torch.tensor(list(mine), dtype=torch.uint8, device=device)
        recv = torch.empty(comm.world * 64, dtype=torch.uint8, device=device)
        comm.dist.all_gather_into_tensor(recv, send, group=comm.group)
        handles = (ctypes.c_ubyte * (64 * comm.world))(*recv.cpu().tolist())
        L.check(lib.nnfac_xchg_attach(self.handle, comm.world, comm.rank, handles))
        base = lib.nnfac_xchg_ptr(self.handle, 0)
        self.tailblk = torch.as_tensor(_RawView(base, (r, self.tpad)), device=device)
        self.inbox = torch.as_tensor(_RawView(base + 4 * self.inbox_off, (self.nslabs, self.r_pad, chunk)), device=device)
        self._scratch = None
        self.send = torch.as_tensor(_RawView(lib.nnfac_xchg_ptr(self.handle, 1), (r, chunk + self.tpad)), device=device)
        comm.dist.barrier(group=comm.group)              # every region is mapped everywhere before anybody posts

    def post(self, phase):
        L.check(L.load_library().nnfac_xchg_post(self.handle, phase, L.stream_ptr()))

    def post_tail(self, vec):
        """post(0) that first writes `vec` (r values) into column 0 of the tail block (one kernel)."""
        L.check(L.load_library().nnfac_xchg_post_tail(self.handle, L.ptr(vec), self.r, self.tpad, 0, L.stream_ptr()))

    def attach_plan(self, plan):
        """The fused passes of `plan` over side 0 that keep their partials write them into the owners' inboxes."""
        slabs, stride = ctypes.c_int(), ctypes.c_int64()
        L.check(L.load_library().nnfac_nmf_plan_set_push(plan.handle, self.handle, self.inbox_off, self.chunk, ctypes.byref(slabs),
                                                         ctypes.byref(stride)))
        assert slabs.value == self.nslabs and stride.value == self.slab_stride, (slabs.value, stride.value, self.nslabs, self.slab_stride)

    def inbox_mu_apply(self, Ft, lo, ncols, floor):
        """mu.py:84-88 for this rank's rows of U from the inbox (local) and the peers' tail blocks -> send buffer."""
        L.check(L.load_library().nnfac_xchg_inbox_mu_apply(self.handle, self.inbox_off, self.nslabs, self.slab_stride, self.chunk, self.tpad,
                                                           L.ptr(Ft), Ft.stride(0), self.r, lo, ncols, float(floor), self.chunk + self.tpad,
                                                           L.stream_ptr()))

    def inbox_sum(self, ncols):
        """The plain sum of the slabs of the inbox -> (r x ncols) (after a kernel that waited for the posts)."""
        out = torch.empty((self.r, ncols), dtype=torch.float32, device=self.device)
        L.check(L.load_library().nnfac_reduce_slabs_f32(L.ctx(self.device), L.ptr(self.inbox), self.chunk, self.nslabs, self.r, self.r_pad,
                                                        ncols, L.ptr(out), out.stride(0), L.stream_ptr()))
        return out

    def scratch(self, r, n):
        if self._scratch is None or self._scratch.numel() < r * n:
            self._scratch = torch.empty(r * n, dtype=torch.float32, device=self.device)
        return self._scratch

    def pull_tail(self, phase, length):
        """Sum over the ranks of the `tail` columns behind column `length` of every rank's buffer `phase` ([r x (length + tpad)])
        -> (r x tail) (after post(phase); waits).  (0, 0): the partial Grams in the tail blocks; (1, chunk): the slices' Grams."""
        out = torch.empty((self.r, self.tail), dtype=torch.float32, device=self.device)
        L.check(L.load_library().nnfac_xchg_pull_tail(self.handle, phase, L.ptr(out), out.stride(0), self.r, length + self.tpad, length,
                                                      self.tail, L.stream_ptr()))
        return out

    def install(self, plan, which, length):
        """All slices straight from the peers' send buffers -> the factor (r x length) and its operand planes in `plan`."""
        out = torch.empty((self.r, length), dtype=torch.float32, device=self.device)
        L.check(L.load_library().nnfac_nmf_plan_set_factor_pulled(plan.handle, which, self.handle, self.chunk, self.chunk + self.tpad,
                                                                  L.ptr(out), out.stride(0), L.stream_ptr()))
        return out

    def close(self):
        try:
            if self.handle:
                torch.cuda.synchronize(self.device)
                L.load_library().nnfac_xchg_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    __del__ = close


class CudaEngine:
    """The device operators one outer iteration is made of, all in libnnfac_b200 (no torch arithmetic)."""

    def __init__(self, X, r, device=None, planes=2):
        self.plan = ops.NMFPlan(X, device).bind_rank(r, planes=planes)

    def set_factor(self, which, Ft):
        self.plan.set_factor(which, Ft)

    def fused(self, side, mode, want_cost, keep_partials=False, cost_out=None, out=None):
        return self.plan.fused(side, mode, want_cost=want_cost, keep_partials=keep_partials, cost_out=cost_out, out=out)

    def mu_finish(self, which, F, den_vec):
        """mu.py:84-88 on the numerator the last fused(which, MODE_MU, keep_partials=True) left in the plan,
        plus the installation of the new factor: one kernel."""
        if self.plan.planes == 3:       # nnfac_nmf_plan_mu_finish writes two planes: update on a copy, then install
            new = self.mu_apply(F, self.plan.reduce(which), den_vec)
            self.set_factor(which, new)
            return new
        return self.plan.mu_finish(which, F, den_vec, mu.epsilon)

    def fused_beta(self, side, beta, want_cost, cost_out=None):
        return self.plan.fused_beta(side, beta, want_cost=want_cost, cost_out=cost_out)

    def mu_finish_beta(self, which, F, beta):
        """mu.py:84-97 from the two partial sets of the last fused_beta(which), plus the installation of the new factor."""
        return self.plan.mu_finish_beta(which, F, gamma_beta(beta), mu.epsilon)

    def cross(self, which, F):
        return self.plan.cross(which, F)

    gram = staticmethod(ops.gram)                      # F (r x len) -> F F^T (nmf.py:407 / :432)

    def solve_install(self, which, UtM, UtU, F, r, sparsity, normalize, result):
        """F <- hals_nnls_acc(UtM, UtU, F) (nmf.py:415 / :440) and F becomes factor `which` of the plan.  One kernel when the
        tensor-core sweep covers the case (it writes the operand planes itself), else solve on a copy + set_factor."""
        sp = 0.0 if sparsity is None else float(sparsity)
        if not normalize and type(self).sweep is CudaEngine.sweep:
            new = self.plan.hals_solve(which, UtM, UtU, F, 100, 0.01, sp, result)   # UtM None: the plan's split-K partials
            if new is not None:
                return new
        if UtM is None:
            UtM = self.plan.reduce(which)
        new = F.clone()
        if self.plan.planes == 3 and not TC_SWEEP_FP32X3 and type(self).sweep is CudaEngine.sweep:
            ops.hals_nnls(UtM, UtU, new, r, 100, 0.01, sp, bool(normalize), False, result, no_tc=True)
        else:
            self.sweep(UtM, UtU, new, r, sparsity, normalize, result)
        self.set_factor(which, new)
        return new

    @staticmethod
    def sweep(UtM, UtU, V, r, sparsity, normalize, result):
        sp = 0.0 if sparsity is None else float(sparsity)
        ops.hals_nnls(UtM, UtU, V, r, 100, 0.01, sp, bool(normalize), False, result)   # nmf.py:415 / :440

    @staticmethod
    def solve_slice(UtM, UtU, F_in, out, r, sparsity, result, comm, lengths):
        """out <- hals_nnls_acc(UtM, UtU, F_in) for this rank's column slice of a solve that spans the group (F_in: strided view
        of the full factor, out: the contiguous send buffer of the all-gather); global stop rule of nnls.py:156."""
        sp = 0.0 if sparsity is None else float(sparsity)
        with comm.collective(lengths):
            if out.shape[1] > 0:
                ops.hals_solve(UtM, UtU, F_in, out, r, 100, 0.01, sp, result)

    def install_gathered(self, which, gathered, length):
        """gathered: [world][r][chunk] slices of the new factor -> the factor (r x length) and all of its operand planes."""
        return self.plan.set_factor_gathered(which, gathered, length)

    @staticmethod
    def mu_apply(F, num, den_vec):
        return ops.mu_apply(F, num, den_vec=den_vec, vec_per_row=True, gamma=1.0, floor=mu.epsilon)   # mu.py:88

    row_sums = staticmethod(ops.row_sums)
    matmul = staticmethod(ops.matmul)

    @staticmethod
    def mu_apply_mat(F, num, den):
        return ops.mu_apply(F, num, den_mat=den, gamma=1.0, floor=mu.epsilon)       # mu.py:89-91

    @staticmethod
    def max_col_abs_sum(F):
        """numpy's matrix 1-norm of F (nmf.py:452)."""
        return ops.norm1(F)

    transpose = staticmethod(ops.transpose)


class FusedNMF:
    events = None   # set to [] to collect (name, start_event, end_event) per phase

    def __init__(self, data, U, V, device=None, group=None, engine=None):
        """data: X (m x n), or this rank's column block X_p when `group` spans several ranks;
        U: m x r (replicated); V: r x n, or this rank's block V_p.  The plan's planes per value follow config.precision
        (3 under "fp32x3", one GPU only)."""
        self.comm = group if isinstance(group, Comm) else Comm(group)
        self.r = int(U.shape[1])
        if engine is None:
            planes = planes_of_precision()
            if planes == 3 and self.comm.world > 1:
                raise NotImplementedError("precision 'fp32x3' covers one GPU (the sharded exchanges write two planes)")
            # a host-resident X goes straight into the plan (upload pipelined with the ingest)
            if isinstance(data, torch.Tensor) and data.is_cuda:
                data = data.to(dtype=torch.float32).contiguous()
            self.eng = CudaEngine(data, self.r, device, planes=planes)
            self.m, self.n = self.eng.plan.m, self.eng.plan.n
            self.device = self.eng.plan.device
            U_dev = L.to_device(U, torch.float32, device)
            V_dev = L.to_device(V, torch.float32, device)
            self._on_gpu = True
        else:
            self.eng = engine
            self.m, self.n = data.shape
            U_dev, V_dev = torch.as_tensor(U), torch.as_tensor(V)
            self.device = U_dev.device
            self._on_gpu = self.device.type == "cuda"
        self.Ut = self.eng.transpose(U_dev)
        self.V = V_dev.clone() if isinstance(V, torch.Tensor) else V_dev
        self.eng.set_factor(0, self.Ut)
        self.eng.set_factor(1, self.V)
        self.hals_stats = torch.zeros((2, 4), dtype=torch.float64, device=self.device)
        self.sweep_log = []
        self._host = torch.zeros(4, dtype=torch.float64)
        if self._on_gpu:
            self._host = self._host.pin_memory()
        self._host_np = self._host.numpy()             # same memory: reading a scalar costs no tensor indexing
        self._dev_scal = torch.zeros(4, dtype=torch.float64, device=self.device)
        # Grams of the single-GPU HALS path are computed on a side stream, under the X pass that precedes their use
        self._side = torch.cuda.Stream(self.device) if self._on_gpu else None
        self._gram = [torch.empty((self.r, self.r), dtype=self.Ut.dtype, device=self.device) for _ in range(2)]
        self._rsum = [torch.empty(self.r, dtype=self.Ut.dtype, device=self.device) for _ in range(2)]
        # exchange buffer of the U side: [cross product or numerator (r x m) | Gram (r x r) or row sums (r)]
        self._xbuf = torch.empty(self.r * self.m + self.r * self.r, dtype=self.Ut.dtype, device=self.device)
        self._usend = None
        self._vlens = self.comm.all_lengths(self.n, self.device)
        self._px = {}
        self._pushing = None
        if self.comm.world > 1 and self._on_gpu and engine is None:
            self.comm.attach_boards(self.device)

    def _phase(self, name):
        from nn_fac.nmf import _Phase
        return _Phase(self, name)

    def _exchange(self, tail):
        """The peer-memory exchange region of this state (tail = r: HALS, partial Gram; tail = 1: MU, partial row sums), or None:
        one rank, CPU stand-in engine, no peer access, NNFAC_PEER_EXCHANGE=0, or slices of U that are not whole 128-row tiles of
        the fused pass (then the NCCL collectives are used)."""
        if (self.comm.world == 1 or not self._on_gpu or not hasattr(self.eng, "plan") or self.comm._boards_device is None
                or os.environ.get("NNFAC_PEER_EXCHANGE", "1") == "0"):
            return None
        if tail not in self._px:
            chunk = self.comm.slice_of(self.m)[0]
            if chunk % 128 != 0:
                return None
            splits = self.eng.plan.info(0)["splits"]
            key = (self.comm.group, L.device_index(self.device), self.r, self.m, chunk, tail, splits)
            if key not in _EXCHANGES:
                _EXCHANGES[key] = PeerExchange(self.comm, self.device, self.r, chunk, tail, splits)
            self._px[tail] = _EXCHANGES[key]
        px = self._px[tail]
        if self._pushing is not px:
            px.attach_plan(self.eng.plan)          # the plan pushes into ONE region at a time (HALS: tail r, MU: tail 1)
            self._pushing = px
        return px

    def _gram_async(self, which, F, out=None):
        """F F^T into `out` (default self._gram[which]) on the side stream (it only reads F, which is final by now); returns a
        function that makes the current stream wait for it."""
        out = self._gram[which] if out is None else out
        if self._side is None:
            self.eng.gram(F, out=out)
            return lambda: out
        main = torch.cuda.current_stream(self.device)
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self.eng.gram(F, out=out)

        def join():
            main.wait_stream(self._side)
            return out
        return join

    def _row_sums_async(self, which, F):
        """Row sums of F (mu.py:85-87 denominators) into self._rsum[which] on the side stream, under the X pass that
        precedes their use; returns the join like _gram_async."""
        if self._side is None:
            return lambda: self.eng.row_sums(F)
        main = torch.cuda.current_stream(self.device)
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self.eng.row_sums(F, out=self._rsum[which])

        def join():
            main.wait_stream(self._side)
            return self._rsum[which]
        return join

    # one outer iteration, given the result of its first pass
    def _apply_hals(self, VMt, sparsity, fixed_modes, normalize, VVt_join=None):
        r, m = self.r, self.m
        Ut, V, comm, eng = self.Ut, self.V, self.comm, self.eng
        if 0 not in fixed_modes:
            with self._phase("gram_U"):
                if comm.world == 1:
                    VVt = VVt_join() if VVt_join is not None else eng.gram(V)      # nmf.py:407
                elif normalize[0]:
                    # partial V_p X_p^T and V_p V_p^T of this column block, summed over the blocks (every rank needs all of
                    # it: a normalised row of U^T spans every slice)
                    xb = self._xbuf
                    xb[:r * m].view(r, m).copy_(VMt)
                    eng.gram(V, out=xb[r * m:].view(r, r))
                    comm.sum_(xb)
                    VMt, VVt = xb[:r * m].view(r, m), xb[r * m:].view(r, r)
                else:
                    # the U solve is split by rows of U: this rank only needs its own columns of the summed V X^T (and the
                    # summed Gram) -> reduce-scatter
                    chunk, lo, hi = comm.slice_of(m)
                    px = self._exchange(r) if VMt is None else None
                    if px is not None:
                        # peer-memory exchange: the fused pass of every rank has already written its partials of MY rows into my
                        # inbox; only the partial Grams (r x r) are pulled.  pull_tail waits for every rank's post.
                        if VVt_join is not None:
                            g = VVt_join()                                         # run() aimed it at the tail block already
                            if g.data_ptr() != px.tailblk.data_ptr():
                                px.tailblk[:, :r].copy_(g)
                        else:
                            eng.gram(V, out=px.tailblk[:, :r])
                        px.post(0)
                        VVt = px.pull_tail(0, 0)
                        VMt_slice = None
                    elif VMt is None:
                        # the pass left its split-K partials in the plan: ONE kernel sums them straight into the send layout of the
                        # reduce-scatter and appends the partial Gram (computed under the pass, on the side stream)
                        gram = VVt_join() if VVt_join is not None else eng.gram(V)
                        recv = comm.reduce_scatter_send(eng.plan.reduce_chunked(0, comm.world, chunk, gram))
                        VMt_slice, VVt = recv[:, :chunk], recv[:, chunk:]
                    else:
                        VMt_slice, VVt = comm.reduce_scatter_columns(VMt, eng.gram(V), chunk)
                        VVt = VVt.contiguous()
            with self._phase("sweep_U"):
                if (comm.world == 1 or normalize[0]) and hasattr(eng, "solve_install"):
                    Ut = eng.solve_install(0, VMt, VVt, Ut, r, sparsity[0], normalize[0], self.hals_stats[0])   # nmf.py:415
                elif comm.world == 1 or normalize[0]:
                    Ut = Ut.clone()
                    eng.sweep(VMt, VVt, Ut, r, sparsity[0], normalize[0], self.hals_stats[0])
                    eng.set_factor(0, Ut)
                elif hasattr(eng, "solve_slice") and self._exchange(r) is not None and VMt is None:
                    # slice solve straight into this rank's send buffer (the partial Gram of the new slice behind it); after the
                    # post the install kernel reads every slice from its owner's send buffer while it builds the operand planes
                    px = self._exchange(r)
                    with comm.collective(comm.slice_lengths(m)):
                        if hi > lo:
                            ops.hals_solve_slabs(px.inbox, chunk, px.nslabs, px.slab_stride, px.r_pad, px.scratch(r, hi - lo), VVt,
                                                 Ut[:, lo:hi], px.send[:, :hi - lo], r, hi - lo, 100, 0.01,
                                                 0.0 if sparsity[0] is None else float(sparsity[0]), self.hals_stats[0])
                    if hi > lo:
                        eng.gram(px.send[:, :hi - lo], out=px.send[:, chunk:chunk + r])
                    else:
                        px.send[:, chunk:chunk + r].zero_()
                    px.post(1)
                    Ut = px.install(eng.plan, 0, m)
                    self._utu_pulled = px.pull_tail(1, chunk)                        # U^T U = sum of the slices' Grams
                elif hasattr(eng, "solve_slice"):
                    # every rank solves its slice of the rows of U straight into the send buffer of the all-gather; the
                    # gathered slices become the new U^T and its operand planes in one kernel
                    send = self._usend if self._usend is not None and self._usend.shape[1] == chunk else None
                    if send is None:
                        send = self._usend = torch.zeros((r, chunk), dtype=Ut.dtype, device=Ut.device)
                    eng.solve_slice(VMt_slice[:, :hi - lo], VVt, Ut[:, lo:hi], send[:, :hi - lo], r, sparsity[0],
                                    self.hals_stats[0], comm, comm.slice_lengths(m))
                    Ut = eng.install_gathered(0, comm.gather_slices(send), m)
                else:
                    Ut = Ut.clone()
                    if hi > lo:
                        eng.sweep(VMt_slice[:, :hi - lo], VVt, Ut[:, lo:hi], r, sparsity[0], False, self.hals_stats[0])
                    comm.gather_columns_(Ut, chunk, lo, hi)
                    eng.set_factor(0, Ut)
        if 1 not in fixed_modes:
            with self._phase("cross_V"):
                pulled = getattr(self, "_utu_pulled", None)                           # sharded: sum of the slices' Grams
                self._utu_pulled = None
                join = self._gram_async(1, Ut) if (self._side is not None and pulled is None) else None    # nmf.py:432, under the X pass
                UtM = eng.cross(1, None)                                              # nmf.py:433
                UtU = pulled if pulled is not None else (join() if join is not None else eng.gram(Ut))
            with self._phase("sweep_V"):
                if hasattr(eng, "solve_install"):
                    with comm.collective(self._vlens):       # the columns of V are spread over the ranks: joint stop rule
                        V = eng.solve_install(1, UtM, UtU, V, r, sparsity[1], normalize[1], self.hals_stats[1])   # nmf.py:440
                elif hasattr(eng, "sweep_collective") and comm.world > 1:
                    V = V.clone()
                    eng.sweep_collective(UtM, UtU, V, r, sparsity[1], self.hals_stats[1], comm)
                    eng.set_factor(1, V)
                else:
                    V = V.clone()
                    eng.sweep(UtM, UtU, V, r, sparsity[1], normalize[1], self.hals_stats[1])
                    eng.set_factor(1, V)
        return Ut, V

    def _apply_mu2(self, VXt, fixed_modes, VVt_join):
        """beta = 2 multiplicative update (mu.py:89-91): U <- U * (X V^T) / (U V V^T), V <- V * (U^T X) / (U^T U V).  The
        denominators never need the model U V: they are small products with the Grams; the numerators are the two cross
        products (first one fused with the cost of the previous iteration)."""
        Ut, V, eng, comm = self.Ut, self.V, self.eng, self.comm
        UtU_pulled = None
        if 0 not in fixed_modes:
            with self._phase("apply_U"):
                if comm.world > 1:
                    # column-sharded: X V^T and V V^T are sums over the ranks.  The partial numerators of MY rows of U are in my
                    # inbox already (pushed by every rank's fused pass); the partial Grams are pulled; every rank updates its own
                    # rows and the install collects the slices (same exchange as the HALS U side)
                    r, m = self.r, self.m
                    px = self._exchange(r)
                    chunk, lo, hi = comm.slice_of(m)
                    g = VVt_join()
                    if g.data_ptr() != px.tailblk.data_ptr():
                        px.tailblk[:, :r].copy_(g)
                    px.post(0)
                    VVt = px.pull_tail(0, 0)                                       # waits for every rank's post
                    if hi > lo:
                        num = px.inbox_sum(hi - lo)
                        den = eng.matmul(VVt, Ut[:, lo:hi])
                        px.send[:, :hi - lo].copy_(eng.mu_apply_mat(Ut[:, lo:hi].contiguous(), num, den))
                        eng.gram(px.send[:, :hi - lo], out=px.send[:, chunk:chunk + r])
                    else:
                        px.send[:, chunk:chunk + r].zero_()
                    px.post(1)
                    Ut = px.install(eng.plan, 0, m)
                    UtU_pulled = px.pull_tail(1, chunk)                            # U^T U = sum of the slices' Grams
                else:
                    den = eng.matmul(VVt_join(), Ut)                               # (V V^T) U^T = (U V V^T)^T
                    Ut = eng.mu_apply_mat(Ut, VXt, den)
                    eng.set_factor(0, Ut)
        if 1 not in fixed_modes:
            with self._phase("pass_V"):
                join = self._gram_async(1, Ut) if UtU_pulled is None else None
                UtX = eng.cross(1, None)
            with self._phase("apply_V"):
                V = eng.mu_apply_mat(V, UtX, eng.matmul(UtU_pulled if UtU_pulled is not None else join(), V))   # (U^T U) V
                eng.set_factor(1, V)
        return Ut, V

    def _apply_mu(self, numU, fixed_modes, den_join=None):
        r, m = self.r, self.m
        Ut, V, comm, eng = self.Ut, self.V, self.comm, self.eng
        if 0 not in fixed_modes:
            with self._phase("apply_U"):
                den = den_join() if den_join is not None else eng.row_sums(V)      # mu.py:85-87
                px = self._exchange(1) if (comm.world > 1 and numU is None) else None
                if px is not None:
                    # peer-memory exchange: the partial numerators of my rows are already in my inbox (written by every rank's
                    # fused pass), the partial row sums of V travel with the post; every rank applies mu.py:84-88 to its own rows
                    # of U and the install kernel collects the slices (four kernels: post with the row sums, update of this
                    # rank's rows, post, pulled install)
                    chunk, lo, hi = comm.slice_of(m)
                    px.post_tail(den)
                    px.inbox_mu_apply(Ut, lo, hi - lo, mu.epsilon)
                    px.post(1)
                    Ut = px.install(eng.plan, 0, m)
                elif comm.world > 1:
                    xb = self._xbuf[:r * m + r]
                    if numU.data_ptr() != xb.data_ptr():
                        xb[:r * m].view(r, m).copy_(numU)
                    xb[r * m:].copy_(den)
                    comm.sum_(xb)
                    numU, den = xb[:r * m].view(r, m), xb[r * m:]
                    Ut = eng.mu_apply(Ut, numU, den)                               # mu.py:84-88
                    eng.set_factor(0, Ut)
                else:
                    Ut = eng.mu_finish(0, Ut, den)                                 # mu.py:84-88 + planes, one kernel
        if 1 not in fixed_modes:
            with self._phase("pass_V"):
                join = self._row_sums_async(1, Ut) if comm.world == 1 else None    # column sums of U under the X pass
                eng.fused(1, MODE_MU, False, keep_partials=True)
            with self._phase("apply_V"):
                V = eng.mu_finish(1, V, join() if join is not None else eng.row_sums(Ut))   # mu.py:27
        return Ut, V

    def _apply_mu_beta(self, beta, fixed_modes):
        """General-beta multiplicative update (mu.py:84-97) from the partials of the first pass: both contractions of each
        factor come out of one pass over X, and the finish kernel divides, raises to gamma and installs."""
        Ut, V, eng = self.Ut, self.V, self.eng
        if 0 not in fixed_modes:
            with self._phase("apply_U"):
                Ut = eng.mu_finish_beta(0, Ut, beta)
        if 1 not in fixed_modes:
            with self._phase("pass_V"):
                eng.fused_beta(1, beta, False)
            with self._phase("apply_V"):
                V = eng.mu_finish_beta(1, V, beta)
        return Ut, V

    def run(self, n_iter_max, tol, update_rule, sparsity=(None, None), fixed_modes=(), normalize=(False, False),
            verbose=False, beta=None):
        """The reference's outer loop (nmf.py:298-324).  Returns (costs, toc)."""
        gen = general_beta(update_rule, beta)
        if gen and self.comm.world > 1:
            raise NotImplementedError("the column-sharded path covers MU with beta = 1 or 2 only")
        mu2 = update_rule == "mu" and beta == 2       # Frobenius MU: cross products + squared residual, like HALS
        if mu2 and self.comm.world > 1:
            px = self._exchange(self.r) if hasattr(self.eng, "plan") else None
            if px is None or 0 in fixed_modes:
                raise NotImplementedError("column-sharded beta = 2 needs the peer-memory exchange (and a free U)")
        mode = MODE_RES if (update_rule == "hals" or mu2) else MODE_MU
        sp = [0.0 if s is None else float(s) for s in sparsity]
        with_sparsity = update_rule == "hals" and (sp[0] != 0.0 or sp[1] != 0.0)
        if self.comm.world > 1 and update_rule == "hals" and normalize[1]:
            raise NotImplementedError("column-sharded HALS cannot normalise the rows of V: a row spans every rank")
        costs, toc = [], []
        tic = time.time()
        done = torch.cuda.Event() if self._on_gpu else None
        # every iteration's solves report into their own slot {eps, cnt, zero row, sweeps} x (U, V)
        stats_log = torch.zeros((n_iter_max + 1, 2, 4), dtype=torch.float64, device=self.device) if (mode == MODE_RES and not mu2) else None
        for it in range(n_iter_max + 1):
            if stats_log is not None:
                self.hals_stats = stats_log[it]
            VVt_join = den_join = None
            if mode == MODE_RES and (self.comm.world == 1 or self._side is not None) and it < n_iter_max and 0 not in fixed_modes \
                    and not (self.comm.world > 1 and normalize[0]):
                # V V^T under the first pass; sharded over peer memory: straight into this rank's tail block (it is free by
                # now: this stream is behind the install of the previous iteration, which waited for every peer's second post,
                # hence for every peer's pull of the partial Grams)
                px = self._exchange(self.r) if (self.comm.world > 1 and mode == MODE_RES and hasattr(self.eng, "plan")) else None
                VVt_join = self._gram_async(0, self.V, out=px.tailblk[:, :self.r] if px is not None else None)
            if mode == MODE_MU and not gen and self.comm.world == 1 and it < n_iter_max and 0 not in fixed_modes:
                den_join = self._row_sums_async(0, self.V)                         # row sums of V under the first pass
            with self._phase("pass_U"):
                # single GPU: the numerator (MU) / cross product (HALS) stays in the plan as split partials, consumed by
                # mu_finish / by the U solve, which adds them itself (nnfac_nmf_plan_hals_solve(UtM = NULL): 0.025 ms less at C2,
                # no reduction kernel).  The V solve (64 columns per CTA, 16+ slabs) was 0.05 ms slower that way: cross_V reduces.
                keep = self.comm.world == 1 and it < n_iter_max and 0 not in fixed_modes and (
                    mode == MODE_MU or (not mu2 and not normalize[0] and hasattr(self.eng, "plan")))
                # sharded HALS: the partials stay in the plan too; the reduce-scatter's send buffer is built from them
                keep = keep or (self.comm.world > 1 and mode == MODE_RES and it < n_iter_max and 0 not in fixed_modes
                                and (mu2 or not normalize[0]) and hasattr(self.eng, "plan"))
                # the cost lands directly in the scalar block that travels to the host
                if gen:
                    # numerator and denominator partials of U's update stay in the plan and the plan object
                    outA = None
                    self.eng.fused_beta(0, beta, True, cost_out=self._dev_scal[0:1])
                elif self.comm.world > 1 and mode == MODE_MU and it < n_iter_max and 0 not in fixed_modes and self._exchange(1) is not None:
                    # sharded MU over peer memory: the fused pass writes the numerator partials into the owners' inboxes
                    outA, _ = self.eng.fused(0, mode, True, keep_partials=True, cost_out=self._dev_scal[0:1])
                elif self.comm.world > 1 and mode == MODE_MU and hasattr(self.eng, "plan"):
                    # sharded MU: the partial numerator lands directly in the exchange buffer (no 16.8 MB copy before the sum)
                    outA, _ = self.eng.fused(0, mode, True, cost_out=self._dev_scal[0:1],
                                             out=self._xbuf[:self.r * self.m].view(self.r, self.m))
                else:
                    outA, _ = self.eng.fused(0, mode, True, keep_partials=keep, cost_out=self._dev_scal[0:1])
            if it > 0:
                self.comm.sum_(self._dev_scal[0:1])
                if with_sparsity:       # nmf.py:449-452: matrix 1-norms of the factors the cost refers to
                    self._dev_scal[1:2].copy_(self.eng.max_col_abs_sum(self.eng.transpose(self.Ut)))
                    self._dev_scal[2:3].copy_(self.eng.max_col_abs_sum(self.V))
                    self.comm.max_(self._dev_scal[2:3])
                self._host.copy_(self._dev_scal, non_blocking=True)
                if done is not None:
                    done.record()
            # launch iteration `it` before looking at the cost of iteration it-1
            if it < n_iter_max:
                if gen:
                    new_Ut, new_V = self._apply_mu_beta(beta, fixed_modes)
                elif mu2:
                    new_Ut, new_V = self._apply_mu2(outA, fixed_modes, VVt_join)
                elif mode == MODE_RES:
                    new_Ut, new_V = self._apply_hals(outA, sparsity, fixed_modes, normalize, VVt_join)
                else:
                    new_Ut, new_V = self._apply_mu(outA, fixed_modes, den_join)
            if it > 0:
                if done is not None:
                    done.synchronize()
                cost = float(self._host_np[0])
                if mu2:
                    cost *= 0.5                         # beta_divergence(., ., 2) = ||X - U V||^2 / 2 (beta_divergence.py:51-52)
                if with_sparsity:
                    cost += 2 * (sp[0] * float(self._host_np[1]) + sp[1] * float(self._host_np[2]))
                toc.append(time.time() - tic)
                costs.append(cost)
                if verbose:
                    if len(costs) == 1:
                        print('Normalized cost function value={}'.format(cost))
                    else:
                        gain = costs[-2] - costs[-1]
                        line = 'Normalized cost function value={}, variation={}.'.format(costs[-1], gain)
                        print(line if gain > 0 else '\033[91m' + line + '\033[0m')
                if len(costs) >= 2 and abs(costs[-2] - costs[-1]) < tol:                 # nmf.py:320
                    if verbose:
                        print('Converged in {} iterations.'.format(len(costs) - 1))
                    # the speculative iteration is dropped: self.Ut / self.V are untouched; put their planes back
                    if it < n_iter_max:
                        self.eng.set_factor(0, self.Ut)
                        self.eng.set_factor(1, self.V)
                    break
            if it == n_iter_max:
                break
            if mode == MODE_RES and not mu2:
                self.sweep_log.append(self.hals_stats[:, 3])       # a view of this iteration's slot of the log: no copy kernel
            self.Ut, self.V = new_Ut, new_V
        return costs, toc

    def factors(self):
        return self.eng.transpose(self.Ut), self.V
