"""NTF multiplicative update at C4 (512 x 512 x 512, rank 32, T = [[A, B, C]] + 0.1 mean rand): it/s of the tensor-core path (the
fused MU pass over the one copy of the tensor as bf16 hi/lo planes, views for modes 1 and 2, no tensor-sized model) against the
CUDA-core path it replaces (NNFAC_NTF_TC=0: K = F krao^T in HBM, the element-wise temporaries, two strided GEMMs per mode and a
model for the cost), for beta in {1, 2, 0, 1.5}.  The two paths alternate in one process (each timing: --warmup iterations, then
--iters timed ones ending in a device synchronise; median of --reps).  Both paths then run --check iterations of ntf() from the
same start and their final objectives are compared.  The fused pass's kernel time comes from torch.profiler in a run of its own,
with its HBM rate at 4 bytes per tensor element (the planes, 512 MiB, do not fit the L2).  The card's name and power limit are
read in the same run.

    python tools/bench_ntf_mu.py [--size 512] [--rank 32] [--warmup 3] [--iters 10] [--reps 3] [--check 10] [--out DIR]

Prints one JSON document (and writes it to DIR/bench_ntf_mu.json with --out)."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nn-fac_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import nn_fac.ntf as ntf  # noqa: E402
from bench_mu_beta import card  # noqa: E402

BETAS = (1, 2, 0, 1.5)
HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU


def make_state(T, F0, tc):
    os.environ["NNFAC_NTF_TC"] = tc
    try:
        return ntf.DeviceNTF(T, F0, torch.float32)
    finally:
        del os.environ["NNFAC_NTF_TC"]


def rate(state, r, beta, warmup, iters):
    args = (r, 1.0, "mu", beta, [None] * 3, [], [False] * 3)
    for _ in range(warmup):
        state.step_async(*args)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        state.step_async(*args)
    torch.cuda.synchronize()
    return iters / (time.perf_counter() - t0)


def objective(T, F0, r, beta, iters, tc):
    os.environ["NNFAC_NTF_TC"] = tc
    try:
        _, costs, _ = ntf.ntf(T, r, init="custom", factors_0=[f.clone() for f in F0], n_iter_max=iters, tol=-1, update_rule="mu",
                              beta=beta, sparsity_coefficients=[None] * 3, fixed_modes=[], normalize=[False] * 3, return_costs=True)
    finally:
        del os.environ["NNFAC_NTF_TC"]
    return costs[-1]


def fused_kernel_us(state, r, beta):
    """Mean device time of the fused pass (tc_fused_kernel) over one profiled iteration, in microseconds."""
    from torch.profiler import ProfilerActivity, profile
    args = (r, 1.0, "mu", beta, [None] * 3, [], [False] * 3)
    state.step_async(*args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        state.step_async(*args)
        torch.cuda.synchronize()
    times = [e.time_range.elapsed_us() for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "tc_fused_kernel" in e.name]
    kernels = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})
    return (sum(times) / len(times) if times else None), len(times), kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--rank", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ntf_mu needs a GPU")
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    n, r = a.size, a.rank
    fs = [torch.rand((n, r), device=dev, generator=g) for _ in range(3)]
    T = torch.einsum("ir,jr,kr->ijk", *fs)
    T += 0.1 * float(T.mean()) * torch.rand((n, n, n), device=dev, generator=g)
    F0 = [f * (1 + 0.3 * torch.rand(f.shape, device=dev, generator=g)) for f in fs]
    del fs
    res = {"shape": [n, n, n, r], "data": "[[A, B, C]] + 0.1 mean rand", "card": card(),
           "timing": {"warmup": a.warmup, "iters": a.iters, "reps": a.reps}, "it_per_s": {}, "median_it_per_s": {}, "speedup": {},
           "objective": {}, "fused_pass": {}}
    for beta in BETAS:
        tag = f"beta={beta}"
        states = {"tensor_core": make_state(T, F0, "1"), "cuda_core": make_state(T, F0, "0")}
        assert states["tensor_core"].direct_cost("mu") and not states["cuda_core"].direct_cost("mu")
        rates = {k: [] for k in states}
        for _ in range(a.reps):                                           # alternate the two paths
            for k, st in states.items():
                rates[k].append(rate(st, r, beta, a.warmup, a.iters))
        res["it_per_s"][tag] = rates
        res["median_it_per_s"][tag] = {k: statistics.median(v) for k, v in rates.items()}
        res["speedup"][tag] = res["median_it_per_s"][tag]["tensor_core"] / res["median_it_per_s"][tag]["cuda_core"]
        us, count, kernels = fused_kernel_us(states["tensor_core"], r, beta)
        entry = {"launches_per_iteration": count, "mean_us": us}
        if us:
            entry["hbm_tb_per_s_at_4_bytes_per_element"] = 4 * n ** 3 / (us * 1e-6) / 1e12
            entry["hbm_fraction"] = 4 * n ** 3 / (us * 1e-6) / HBM_BYTES_PER_S
        else:
            entry["kernels_seen"] = kernels
        res["fused_pass"][tag] = entry
        del states
        torch.cuda.empty_cache()
        c_tc = objective(T, F0, r, beta, a.check, "1")
        c_cc = objective(T, F0, r, beta, a.check, "0")
        res["objective"][tag] = {"iterations": a.check, "tensor_core": c_tc, "cuda_core": c_cc, "rel_diff": abs(c_tc - c_cc) / abs(c_cc)}
        torch.cuda.empty_cache()
        print(json.dumps({tag: [res["median_it_per_s"][tag], res["fused_pass"][tag], res["objective"][tag]]}), flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_ntf_mu.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
