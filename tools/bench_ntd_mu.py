"""NTD multiplicative update at C5 (256^3, core 32^3) and at 512^3 / 32^3 (T = G x_n F_n + 0.1 mean rand): it/s of the tensor-core
path (one copy of the tensor as bf16 hi/lo planes, views for the other modes and for the core update's contraction over mode 0, no
tensor-sized temporary) against the CUDA-core path (NNFAC_NTD_TC=0: the model K in HBM, the element-wise terms, strided GEMMs), for
beta in {1, 2, 0, 1.5}.  The two paths alternate in one process (each timing: --warmup iterations, then --iters timed ones ending
in a device synchronise; median of --reps).  Both paths then run --check iterations of ntd() from the same start and their final
objectives are compared.  The tensor-core passes' kernel time (tc_fused_kernel, tc_cross_kernel) comes from torch.profiler in a run
of its own; the bytes the plans hold are summed from their workspaces.  The card's name and power limit are read in the same run.

    python tools/bench_ntd_mu.py [--sizes 256,512] [--rank 32] [--warmup 3] [--iters 10] [--reps 3] [--check 10] [--out DIR]

Prints one JSON document (and writes it to DIR/bench_ntd_mu.json with --out)."""
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

import nn_fac.ntd as ntd  # noqa: E402
from bench_mu_beta import card  # noqa: E402

BETAS = (1, 2, 0, 1.5)


def make_state(T, G0, F0, tc):
    os.environ["NNFAC_NTD_TC"] = tc
    try:
        return ntd.DeviceNTD(T, G0, F0, torch.float32)
    finally:
        del os.environ["NNFAC_NTD_TC"]


def rate(state, beta, warmup, iters):
    args = (beta, [], [False] * 4, None)
    state.invalidate()
    for _ in range(warmup):
        state.step_mu_async(*args)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        state.step_mu_async(*args)
    torch.cuda.synchronize()
    return iters / (time.perf_counter() - t0)


def objective(T, G0, F0, beta, iters, tc):
    os.environ["NNFAC_NTD_TC"] = tc
    try:
        _, _, costs, _ = ntd.ntd(T, [int(s) for s in G0.shape], init="custom", core_0=G0.clone(), factors_0=[f.clone() for f in F0],
                                 n_iter_max=iters, tol=0, update_rule="mu", beta=beta, sparsity_coefficients=[None] * 4, fixed_modes=[],
                                 normalize=[False] * 4, return_costs=True)
    finally:
        del os.environ["NNFAC_NTD_TC"]
    return costs[-1]


def plan_bytes(state):
    held = 0
    for p in state.plans + [state.core_plan]:
        held += p._workspace.numel() + (0 if p._den is None else p._den.numel() * 4) + (0 if p._xf32 is None else p._xf32.numel())
    return held


def pass_kernels_us(state, beta):
    """Device time of the tensor-core passes over the tensor (tc_fused_kernel / tc_cross_kernel) in one profiled iteration."""
    from torch.profiler import ProfilerActivity, profile
    args = (beta, [], [False] * 4, None)
    state.step_mu_async(*args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        state.step_mu_async(*args)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    out = {}
    for key in ("tc_fused_kernel", "tc_cross_kernel"):
        t = [e.time_range.elapsed_us() for e in ev if key in e.name]
        out[key] = {"launches_per_iteration": len(t), "total_us": sum(t)}
    out["all_kernels_us"] = sum(e.time_range.elapsed_us() for e in ev)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="256,512")
    ap.add_argument("--rank", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ntd_mu needs a GPU")
    dev = torch.device("cuda", 0)
    rc = a.rank
    res = {"data": "G x_n F_n + 0.1 mean rand", "card": card(), "timing": {"warmup": a.warmup, "iters": a.iters, "reps": a.reps},
           "results": {}}
    for n in (int(s) for s in a.sizes.split(",")):
        g = torch.Generator(device=dev).manual_seed(11)
        G = torch.rand((rc,) * 3, generator=g, device=dev)
        Fs = [torch.rand((n, rc), generator=g, device=dev) for _ in range(3)]
        T = torch.einsum("abc,ia,jb,kc->ijk", G, *Fs)
        T.add_(torch.rand((n,) * 3, generator=g, device=dev), alpha=0.1 * float(T.mean()))
        G0 = torch.rand((rc,) * 3, generator=g, device=dev)
        F0 = [torch.rand((n, rc), generator=g, device=dev) for _ in range(3)]
        del G, Fs
        shape_key = f"{n}^3 core {rc}^3"
        out = res["results"][shape_key] = {}
        for beta in BETAS:
            tag = f"beta={beta}"
            states = {"tensor_core": make_state(T, G0, F0, "1"), "cuda_core": make_state(T, G0, F0, "0")}
            assert states["tensor_core"].plans is not None and states["cuda_core"].plans is None
            rates = {k: [] for k in states}
            for _ in range(a.reps):                                       # alternate the two paths
                for k, st in states.items():
                    rates[k].append(rate(st, beta, a.warmup, a.iters))
            med = {k: statistics.median(v) for k, v in rates.items()}
            entry = {"it_per_s": rates, "median_it_per_s": med, "speedup": med["tensor_core"] / med["cuda_core"],
                     "plan_bytes_per_element": plan_bytes(states["tensor_core"]) / T.numel(),
                     "passes": pass_kernels_us(states["tensor_core"], beta)}
            del states
            torch.cuda.empty_cache()
            c_tc = objective(T, G0, F0, beta, a.check, "1")
            c_cc = objective(T, G0, F0, beta, a.check, "0")
            entry["objective"] = {"iterations": a.check, "tensor_core": c_tc, "cuda_core": c_cc, "rel_diff": abs(c_tc - c_cc) / abs(c_cc)}
            torch.cuda.empty_cache()
            out[tag] = entry
            print(json.dumps({shape_key: {tag: [med, entry["speedup"], entry["objective"]["rel_diff"]]}}), flush=True)
        del T, G0, F0
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_ntd_mu.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
