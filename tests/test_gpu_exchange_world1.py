"""Device kernels of the column-sharded path, checked on one GPU as a group of one.

At world size 1 an exchange region (nnfac_xchg_*) and the sweep boards (nnfac_ctx_board_*) map this process' own memory and open
no IPC handle, so every kernel of the sharded U side -- chunked reduction, gathered / pulled install, the push layout of the fused
pass, the tail pull, the multi-slab HALS solve and the collective stop rule -- runs here and is compared bit for bit with its
single-GPU twin (or with float64).

Every call that waits (pull_tail, inbox_mu_apply, set_factor_pulled) is issued after this rank's own post of that phase: a wait with
no matching post would spin until the kernel traps."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _lib():
    from nn_fac import _lib as L
    return L, L.load_library()


@contextlib.contextmanager
def _region(stage_floats, send_floats):
    """An exchange region of one rank: created, attached as rank 0 of 1 (the 64 handle bytes are never read), destroyed."""
    L, lib = _lib()
    h = ctypes.c_void_p()
    L.check(lib.nnfac_xchg_create(L.ctx(), int(stage_floats), int(send_floats), ctypes.byref(h)))
    try:
        L.check(lib.nnfac_xchg_attach(h, 1, 0, (ctypes.c_ubyte * 64)()))
        yield h
    finally:
        torch.cuda.synchronize()
        lib.nnfac_xchg_destroy(h)


def _view(h, which, shape):
    """The stage (0) or send (1) buffer of a region as a float32 tensor of `shape` (from its start)."""
    from nn_fac._fast import _RawView
    L, lib = _lib()
    return torch.as_tensor(_RawView(lib.nnfac_xchg_ptr(h, which), shape), device="cuda")


def _plan_pair(X, Ut, V, r):
    from nn_fac import _ops as ops
    plans = [ops.NMFPlan(_dev(X)).bind_rank(r) for _ in range(2)]
    for p in plans:
        p.set_factor(0, Ut)
        p.set_factor(1, V)
    return plans


def _problem(m, n, r, seed):
    rng = np.random.RandomState(seed)
    X = (rng.rand(m, r) @ rng.rand(r, n) + 0.3 * rng.rand(m, n)).astype(np.float32)
    Ut = _dev((rng.rand(r, m) + 0.05).astype(np.float32))
    V = _dev((rng.rand(r, n) + 0.05).astype(np.float32))
    return X, Ut, V


# ---------------------------------------------------------------------------------------------
# chunked reduction (send layout of a reduce-scatter)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("side", [0, 1])
def test_reduce_chunked_equals_reduce(side):
    """Column `row` of reduce(side) lands in out[row // chunk][k][row % chunk], columns at or beyond R are 0, the tail is copied
    behind every chunk: bit for bit, one slab and three, R a multiple of chunk and not."""
    from nn_fac import _ops as ops
    m, n, r = 1536, 2304, 40
    X, Ut, V = _problem(m, n, r, 5)
    plan = ops.NMFPlan(_dev(X)).bind_rank(r)
    plan.set_factor(0, Ut)
    plan.set_factor(1, V)
    assert plan.info(side)["splits"] > 1            # the reduction has split-K partials to add
    plan.fused(side, 0, keep_partials=True)
    full = plan.reduce(side)
    R = full.shape[1]
    rng = np.random.RandomState(side)
    for slabs in (1, 3):
        for chunk in (R // slabs, -(-R // slabs) + 37):
            assert (R % chunk == 0) == (chunk == R // slabs)
            for tail in (None, _dev(rng.rand(r, r).astype(np.float32)), _dev(rng.rand(r, 3).astype(np.float32))):
                out = plan.reduce_chunked(side, slabs, chunk, tail)
                t = 0 if tail is None else tail.shape[1]
                assert out.shape == (slabs, r, chunk + t)
                want = torch.zeros((r, slabs * chunk), dtype=torch.float32, device="cuda")
                want[:, :R] = full
                assert torch.equal(out[:, :, :chunk], want.view(r, slabs, chunk).permute(1, 0, 2)), (slabs, chunk, t)
                if tail is not None:
                    assert torch.equal(out[:, :, chunk:], tail.unsqueeze(0).expand(slabs, r, t)), (slabs, chunk, t)


# ---------------------------------------------------------------------------------------------
# install from gathered slices
# ---------------------------------------------------------------------------------------------
def test_set_factor_gathered_equals_set_factor():
    """[slices][r][chunk] with a ragged last slice (its padding holds large values that must not be read) -> the factor and its
    operand planes: the following cross products and fused passes are bit-identical to those after set_factor."""
    m, n, r = 1000, 1300, 24
    X, Ut, V = _problem(m, n, r, 7)
    plain, gathered = _plan_pair(X, Ut, V, r)
    for which, F in ((0, Ut), (1, V)):
        length = F.shape[1]
        slices = 3
        chunk = -(-length // slices) + 5
        assert slices * chunk > length
        new = F * 0.75 + 0.01                           # a different factor, installed both ways
        plain.set_factor(which, new)
        G = torch.full((slices, r, chunk), 1e30, dtype=torch.float32, device="cuda")
        for s in range(slices):
            lo, hi = s * chunk, min((s + 1) * chunk, length)
            if hi > lo:
                G[s, :, :hi - lo] = new[:, lo:hi]
        Ft = gathered.set_factor_gathered(which, G, length)
        assert torch.equal(Ft, new)
        assert torch.equal(plain.cross(which, None), gathered.cross(which, None))
        for side in (0, 1):
            for mode in (0, 1):
                a, ca = plain.fused(side, mode)
                b, cb = gathered.fused(side, mode)
                assert torch.equal(a, b) and torch.equal(ca, cb), (which, side, mode)


# ---------------------------------------------------------------------------------------------
# HALS solve whose right-hand side is a sum of slabs
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nslabs", [1, 4, 7])
@pytest.mark.parametrize("r,n", [(40, 5000), (96, 60000)])
def test_hals_solve_slabs_equals_solve_of_the_slab_sum(r, n, nslabs):
    """nnfac_hals_solve_slabs_f32 against hals_solve on nnfac_reduce_slabs_f32 of the same slabs: same V, same result vector.  The
    padding rows r <= k < r_pad and columns n <= c < ld of every slab hold large values that must be ignored.  (40, 5000): the
    tensor-core sweep adds the slabs; (96, 60000): more columns per SM than the sweep keeps, the slabs are summed into scratch."""
    from nn_fac import _ops as ops
    L, lib = _lib()
    rng = np.random.RandomState(r + n + nslabs)
    r_pad = -(-(r + 1) // 16) * 16
    ld = -(-n // 128) * 128 + (128 if n % 128 == 0 else 0)
    U = rng.rand(2 * r + 5, r)
    G = (U.T @ U).astype(np.float32)
    B = U.T @ (U @ rng.rand(r, n) + 0.1 * rng.rand(2 * r + 5, n))
    w = rng.rand(nslabs) + 0.2
    w /= w.sum()
    slabs = np.full((nslabs, r_pad, ld), 1e30, dtype=np.float32)
    for s in range(nslabs):
        slabs[s, :r, :n] = (B * w[s] * (1 + 0.1 * rng.rand(r, n))).astype(np.float32)
    slabs_d, G_d = _dev(slabs), _dev(G)
    V0 = _dev(rng.rand(r, n).astype(np.float32))
    total = torch.empty((r, n), dtype=torch.float32, device="cuda")
    L.check(lib.nnfac_reduce_slabs_f32(L.ctx(), L.ptr(slabs_d), ld, nslabs, r, r_pad, n, L.ptr(total), total.stride(0), L.stream_ptr()))
    np.testing.assert_allclose(total.cpu().numpy(), slabs[:, :r, :n].astype(np.float64).sum(axis=0), rtol=1e-6)
    scratch = torch.full((r * n,), 7.0, dtype=torch.float32, device="cuda")
    Va = torch.empty_like(V0)
    ra = torch.zeros(4, dtype=torch.float64, device="cuda")
    ops.hals_solve_slabs(slabs_d, ld, nslabs, r_pad * ld, r_pad, scratch, G_d, V0, Va, r, n, 100, 0.01, 0.0, ra)
    Vb = torch.empty_like(V0)
    rb = torch.zeros(4, dtype=torch.float64, device="cuda")
    ops.hals_solve(total, G_d, V0, Vb, r, 100, 0.01, 0.0, rb)
    assert torch.equal(ra, rb), (ra, rb)
    assert torch.equal(Va, Vb)
    assert 2 <= int(ra[1].item()) <= 101 and (Va >= 0).all()


# ---------------------------------------------------------------------------------------------
# PUSH layout: the fused pass writes its partials into the inbox of an exchange region
# ---------------------------------------------------------------------------------------------
def test_set_push_inbox_equals_plan_partials():
    """After fused(0, mode, keep_partials=True) into the inbox: inbox_mu_apply gives the bits of mu_finish, hals_solve_slabs the
    bits of plan.hals_solve(0, None, ...), reduce_slabs_f32 the bits of plan.reduce(0); set_push(None) restores the plain pass.
    A zero row of X gives a zero numerator: inbox_mu_apply writes the floor there."""
    from nn_fac import _ops as ops
    L, lib = _lib()
    m, n, r = 1000, 4096, 40
    X, Ut, V = _problem(m, n, r, 11)
    X[7] = 0.0
    push, ref = _plan_pair(X, Ut, V, r)
    splits = push.info(0)["splits"]
    assert splits > 1
    chunk = -(-m // 128) * 128
    r_pad = -(-r // 16) * 16
    tpad = 4
    inbox_off = r * tpad
    nslabs = splits
    with _region(inbox_off + nslabs * r_pad * chunk, r * (chunk + tpad)) as h:
        got_slabs, got_stride = ctypes.c_int(), ctypes.c_int64()
        L.check(lib.nnfac_nmf_plan_set_push(push.handle, h, inbox_off, chunk, ctypes.byref(got_slabs), ctypes.byref(got_stride)))
        assert got_slabs.value == nslabs and got_stride.value == r_pad * chunk
        stage = _view(h, 0, (inbox_off + nslabs * r_pad * chunk,))
        inbox = stage[inbox_off:].view(nslabs, r_pad, chunk)
        send = _view(h, 1, (r, chunk + tpad))

        # beta = 1: the numerator partials go to the inbox, the row sums of V travel in column 0 of the tail block
        den = ops.row_sums(V)
        push.fused(0, 1, want_cost=False, keep_partials=True)
        L.check(lib.nnfac_xchg_post_tail(h, L.ptr(den), r, tpad, 0, L.stream_ptr()))
        L.check(lib.nnfac_xchg_inbox_mu_apply(h, inbox_off, nslabs, r_pad * chunk, chunk, tpad, L.ptr(Ut), Ut.stride(0), r, 0, m, 1e-12,
                                              chunk + tpad, L.stream_ptr()))
        ref.fused(0, 1, want_cost=False, keep_partials=True)
        want = ref.mu_finish(0, Ut, den, 1e-12)
        ref.set_factor(0, Ut)
        assert torch.equal(send[:, :m], want)
        assert (send[:, 7] == np.float32(1e-12)).all()
        total = torch.empty((r, m), dtype=torch.float32, device="cuda")
        L.check(lib.nnfac_reduce_slabs_f32(L.ctx(), L.ptr(inbox), chunk, nslabs, r, r_pad, m, L.ptr(total), m, L.stream_ptr()))
        ref.fused(0, 1, want_cost=False, keep_partials=True)
        assert torch.equal(total, ref.reduce(0))

        # HALS: the cross-product partials of the residual pass, solved straight from the inbox
        G = ops.gram(V)
        push.fused(0, 0, keep_partials=True)
        Va = torch.empty_like(Ut)
        ra = torch.zeros(4, dtype=torch.float64, device="cuda")
        ops.hals_solve_slabs(inbox, chunk, nslabs, r_pad * chunk, r_pad, torch.empty(r * m, device="cuda"), G, Ut, Va, r, m, 100, 0.01,
                             0.0, ra)
        ref.fused(0, 0, keep_partials=True)
        rb = torch.zeros(4, dtype=torch.float64, device="cuda")
        Vb = ref.hals_solve(0, None, G, Ut, 100, 0.01, 0.0, rb)
        assert Vb is not None
        assert torch.equal(ra, rb) and torch.equal(Va, Vb)
        ref.set_factor(0, Ut)
        L.check(lib.nnfac_reduce_slabs_f32(L.ctx(), L.ptr(inbox), chunk, nslabs, r, r_pad, m, L.ptr(total), m, L.stream_ptr()))
        ref.fused(0, 0, keep_partials=True)
        assert torch.equal(total, ref.reduce(0))

        # switched off: the partials stay in the plan again
        L.check(lib.nnfac_nmf_plan_set_push(push.handle, None, 0, 0, None, None))
        before = inbox.clone()
        push.fused(0, 1, want_cost=False, keep_partials=True)
        ref.fused(0, 1, want_cost=False, keep_partials=True)
        assert torch.equal(push.mu_finish(0, Ut, den, 1e-12), ref.mu_finish(0, Ut, den, 1e-12))
        assert torch.equal(inbox, before)


# ---------------------------------------------------------------------------------------------
# tail pull (post_tail / post + pull_tail), set_factor_pulled
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("phase", [0, 1])
def test_pull_tail_returns_the_posted_tail(phase):
    """Phase 0: the row sums of V, posted by post_tail into column 0 of the tail block [r x tpad] (tail = 1).  Phase 1: an r x r
    Gram behind the chunk of the send buffer [r x (chunk + tpad)] (col = chunk, tail = r).  Everything around the tail holds large
    values that must not be read; pull_tail returns the posted values bit for bit and writes nothing beyond `tail` columns."""
    L, lib = _lib()
    r, chunk = 22, 640
    tpad = -(-r // 4) * 4
    assert tpad > r                                                   # a padding column in the phase-1 tail
    rng = np.random.RandomState(phase)
    with _region(r * tpad, r * (chunk + tpad)) as h:
        if phase == 0:
            pitch, col, tail = tpad, 0, 1
            want = _dev((rng.rand(r, 1) + 0.5).astype(np.float32))
            stage = _view(h, 0, (r, tpad))
            stage.fill_(1e30)
            L.check(lib.nnfac_xchg_post_tail(h, L.ptr(want), r, tpad, 0, L.stream_ptr()))
        else:
            pitch, col, tail = chunk + tpad, chunk, r
            want = _dev(rng.rand(r, r).astype(np.float32))
            send = _view(h, 1, (r, pitch))
            send.fill_(1e30)
            send[:, chunk:chunk + r].copy_(want)
            L.check(lib.nnfac_xchg_post(h, 1, L.stream_ptr()))
        out = torch.full((r, tail + 3), 5.0, dtype=torch.float32, device="cuda")
        L.check(lib.nnfac_xchg_pull_tail(h, phase, L.ptr(out), out.stride(0), r, pitch, col, tail, L.stream_ptr()))
        assert torch.equal(out[:, :tail], want)
        assert (out[:, tail:] == 5.0).all()


def test_set_factor_pulled_equals_set_factor():
    """The factor read from the (own) send buffer after post(1), its padding holding large values: the factor and the operand
    planes equal those of set_factor (cross products and fused passes bit-identical)."""
    L, lib = _lib()
    m, n, r = 1000, 1300, 24
    X, Ut, V = _problem(m, n, r, 13)
    plain, pulled = _plan_pair(X, Ut, V, r)
    tpad = 4
    chunk = -(-max(m, n) // 128) * 128
    pitch = chunk + tpad
    with _region(r * 8, r * pitch) as h:
        send = _view(h, 1, (r, pitch))
        for which, F in ((0, Ut), (1, V)):
            length = F.shape[1]
            new = F * 0.5 + 0.02
            send.fill_(1e30)
            send[:, :length].copy_(new)
            plain.set_factor(which, new)
            L.check(lib.nnfac_xchg_post(h, 1, L.stream_ptr()))
            out = torch.empty((r, length), dtype=torch.float32, device="cuda")
            L.check(lib.nnfac_nmf_plan_set_factor_pulled(pulled.handle, which, h, chunk, pitch, L.ptr(out), out.stride(0), L.stream_ptr()))
            assert torch.equal(out, new)
            assert torch.equal(plain.cross(which, None), pulled.cross(which, None))
            for side in (0, 1):
                for mode in (0, 1):
                    a, ca = plain.fused(side, mode)
                    b, cb = pulled.fused(side, mode)
                    assert torch.equal(a, b) and torch.equal(ca, cb), (which, side, mode)


# ---------------------------------------------------------------------------------------------
# collective stop rule of the tensor-core sweep, group of one
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r,n", [(64, 8192), (40, 3000), (128, 12000)])
def test_collective_hals_on_a_group_of_one_equals_the_plain_solve(r, n):
    """A solve announced as one slice of a joint solve over a group of one runs the board protocol (every CTA posts its partial
    on the board, sums the board) and must execute the sweeps of the plain solve: same V, same result vector, for both stop-test
    variants, through ops.hals_nnls and through the plan's solve."""
    from nn_fac import _ops as ops
    L, lib = _lib()
    ctx = L.ctx()
    g = torch.Generator(device="cuda")
    g.manual_seed(r + n)
    m = 2 * r + 5
    U = torch.rand((m, r), generator=g, device="cuda")
    G = (U.T @ U).contiguous()
    b = (G @ torch.rand((r, n), generator=g, device="cuda") + 0.1 * torch.rand((r, n), generator=g, device="cuda")).contiguous()
    V0 = torch.rand((r, n), generator=g, device="cuda")
    X = torch.rand((m, n), generator=g, device="cuda")
    handle = (ctypes.c_ubyte * 64)()
    L.check(lib.nnfac_ctx_board_export(ctx, handle))
    L.check(lib.nnfac_ctx_board_attach(ctx, 1, 0, handle))
    lengths = (ctypes.c_int64 * 1)(n)

    def solves():
        V = V0.clone()
        st = ops.hals_nnls(b, G, V, r, 100, 0.01, 0.0, False, False).clone()
        plan = ops.NMFPlan(X).bind_rank(r)
        plan.set_factor(0, U.T.contiguous())
        res = torch.zeros(4, dtype=torch.float64, device="cuda")
        W = plan.hals_solve(1, b, G, V0, 100, 0.01, 0.0, res)
        assert W is not None
        return V, st, W, res

    out = {}
    try:
        for variant in (0, 2):
            L.check(lib.nnfac_ctx_sweep_variant(ctx, variant))
            out[variant, False] = solves()
            L.check(lib.nnfac_ctx_collective(ctx, 1, lengths))
            try:
                out[variant, True] = solves()
            finally:
                L.check(lib.nnfac_ctx_collective(ctx, 0, None))
    finally:
        L.check(lib.nnfac_ctx_sweep_variant(ctx, -1))
    for variant in (0, 2):
        for a, c in zip(out[variant, False], out[variant, True]):
            assert torch.equal(a, c), variant
    assert 2 <= int(out[0, False][1][1].item()) <= 101
