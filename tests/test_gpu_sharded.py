"""The column-sharded path on real GPUs (needs >= 2 visible GPUs; skipped otherwise): the U-side exchange in its two forms --
"push" (default: the fused pass writes its partials into the owners' inboxes over NVLink, nnfac_nmf_plan_set_push) and "nccl"
(NNFAC_PEER_EXCHANGE=0: reduce-scatter / all-gather / all-reduce) --, slice solves with the cross-GPU stop scalar (peer-mapped
boards), the pulled one-kernel install.
The sharded run must reproduce the single-GPU run of the same problem: same sweep counts in every solve, objectives to 1e-6."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir, m, n, r, iters, exchange="push"):
    if exchange == "nccl":
        os.environ["NNFAC_PEER_EXCHANGE"] = "0"
    for p in (ROOT, os.path.join(ROOT, "nn-fac_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    from nn_fac import _fast, _ops as ops
    from nn_fac.sharded import column_block, compute_nmf_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        lo, hi = column_block(n, world, rank)

        def block(c0, c1):
            X = ops.philox_uniform(m, r, seed=9, stream_id=0) @ ops.philox_uniform(r, c1 - c0, col0=c0, seed=9, stream_id=1)
            ops.philox_uniform(m, c1 - c0, col0=c0, seed=9, stream_id=2, scale=r / 4.0, out=X, accumulate=True)
            return X, ops.philox_uniform(m, r, seed=9, stream_id=3), ops.philox_uniform(r, c1 - c0, col0=c0, seed=9, stream_id=4)
        res = {}
        for rule, beta in (("hals", 2), ("mu", 1), ("mu2", 2)):
            if rule == "mu" and r > 64:
                continue
            if rule == "mu2" and exchange != "push":          # the sharded beta = 2 update needs the peer-memory exchange
                continue
            tag, rule = rule, rule.rstrip("2")
            X, U0, V0 = block(lo, hi)
            st = _fast.FusedNMF(X, U0, V0, group=dist.group.WORLD)
            costs = st.run(iters, 0.0, rule, beta=beta)[0]
            res[tag + "_costs"] = np.array(costs)
            res[tag + "_sweeps"] = np.array([t.cpu().numpy() for t in st.sweep_log])
            U, V = st.factors()
            res[tag + "_U"], res[tag + "_V"] = U.cpu().numpy(), V.cpu().numpy()
            del st
            # the public entry point with host arrays
            out = compute_nmf_sharded(X.cpu().numpy(), r, U0.cpu().numpy(), V0.cpu().numpy(), n_iter_max=2, tol=0, update_rule=rule,
                                      beta=beta, return_costs=True)
            np.testing.assert_allclose(out[2], costs[:2], rtol=1e-6)
            if rank == 0:
                X, U0, V0 = block(0, n)
                one = _fast.FusedNMF(X, U0, V0)
                res[tag + "_costs_1"] = np.array(one.run(iters, 0.0, rule, beta=beta)[0])
                res[tag + "_sweeps_1"] = np.array([t.cpu().numpy() for t in one.sweep_log])
                U1, V1 = one.factors()
                res[tag + "_U_1"], res[tag + "_V_1"] = U1.cpu().numpy(), V1.cpu().numpy()
                del one
            dist.barrier()
        res["cols"] = np.array([lo, hi])
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("m,n,r,exchange", [(4096, 2048, 64, "push"), (6000, 1500, 40, "push"), (8192, 2048, 128, "push"),
                                            (4096, 2048, 64, "nccl")])
def test_two_gpus_reproduce_one_gpu(tmp_path, m, n, r, exchange):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    iters = 6
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), m, n, r, iters, exchange), nprocs=2, join=True)
    ranks = [dict(np.load(os.path.join(str(tmp_path), f"rank{k}.npz"))) for k in range(2)]
    for rule in ("hals", "mu", "mu2"):
        if rule + "_costs" not in ranks[0]:
            continue
        np.testing.assert_array_equal(ranks[0][rule + "_costs"], ranks[1][rule + "_costs"])      # every rank sees the same objective
        np.testing.assert_array_equal(ranks[0][rule + "_U"], ranks[1][rule + "_U"])              # U is replicated, bit for bit
        np.testing.assert_allclose(ranks[0][rule + "_costs"], ranks[0][rule + "_costs_1"], rtol=1e-6)
        V = np.concatenate([ranks[0][rule + "_V"], ranks[1][rule + "_V"]], axis=1)
        if rule == "hals":
            # the stop test of nnls.py:156 runs on the squared steps of ALL columns: same sweeps as on one GPU
            np.testing.assert_array_equal(ranks[0]["hals_sweeps"], ranks[0]["hals_sweeps_1"])
            np.testing.assert_array_equal(ranks[0]["hals_sweeps"], ranks[1]["hals_sweeps"])
        for got, want in ((ranks[0][rule + "_U"], ranks[0][rule + "_U_1"]), (V, ranks[0][rule + "_V_1"])):
            assert np.linalg.norm(got - want) <= 1e-3 * np.linalg.norm(want)          # fp32 sums grouped differently
