"""General-beta MU at C2 (65536 x 8192, rank 64, X = W H + 0.1 mean(W H) rand): it/s of the tensor-core pass (FusedNMF) for
beta in {0, 0.5, 1.5, 3} against the CUDA-core path it replaces (nmf.DeviceNMF: K = U V in HBM, two element-wise temporaries, four
strided GEMMs and a separate cost pass; still the path for rank > 64), with MU beta = 1 (fused) as the yardstick.  The paths
alternate in one process after warm-up (median of --reps); the phase times of one iteration come from FusedNMF.events (CUDA
events); both paths run --check iterations from the same start and their final objectives are compared.  The card's name and
power limit are read in the same run.

    python tools/bench_mu_beta.py [--iters 20] [--cc-iters 4] [--reps 3] [--check 10] [--out DIR]

Prints one JSON document (and writes it to DIR/bench_mu_beta.json with --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nn-fac_b200"))
import torch  # noqa: E402

import nn_fac.nmf as nmf  # noqa: E402
from nn_fac import _fast  # noqa: E402

BETAS = (0, 0.5, 1.5, 3)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def timed(fn, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return iters / (time.perf_counter() - t0)


def cuda_core_steps(st, beta, k):
    cost = None
    for _ in range(k):
        cost = st.step("mu", beta, [None, None], [], [False, False])
    return cost


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=65536)
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--r", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--cc-iters", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mu_beta needs a GPU")
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    m, n, r = a.m, a.n, a.r
    X = torch.rand((m, r), device=dev, generator=g) @ torch.rand((r, n), device=dev, generator=g)
    X += 0.1 * float(X.mean()) * torch.rand((m, n), device=dev, generator=g)
    U0 = torch.rand((m, r), device=dev, generator=g)
    V0 = torch.rand((r, n), device=dev, generator=g)
    res = {"shape": [m, n, r], "data": "W H + 0.1 mean(W H) rand", "iters_per_timing": {"tensor_core": a.iters, "cuda_core": a.cc_iters},
           "card": card(), "it_per_s": {}, "median_it_per_s": {}, "phase_ms": {}, "objective": {}}
    for beta in (1,) + BETAS:
        tag = f"beta={beta}"
        tc = _fast.FusedNMF(X, U0, V0)
        tc.run(3, 0.0, "mu", beta=beta)                                  # warm-up
        cc = None
        if beta != 1:
            cc = nmf.DeviceNMF(X, U0, V0, torch.float32)
            cuda_core_steps(cc, beta, 1)
        rates = {"tensor_core": [], "cuda_core": []}
        for _ in range(a.reps):                                           # alternate the two paths
            rates["tensor_core"].append(timed(lambda: tc.run(a.iters, 0.0, "mu", beta=beta), a.iters))
            if cc is not None:
                rates["cuda_core"].append(timed(lambda: cuda_core_steps(cc, beta, a.cc_iters), a.cc_iters))
        if cc is None:
            del rates["cuda_core"]
        res["it_per_s"][tag] = rates
        res["median_it_per_s"][tag] = {k: statistics.median(v) for k, v in rates.items()}
        tc.events = []                                                    # per-phase device times, in a run of their own
        tc.run(a.iters, 0.0, "mu", beta=beta)
        torch.cuda.synchronize()
        acc = {}
        for name, e0, e1 in tc.events:
            acc[name] = acc.get(name, 0.0) + e0.elapsed_time(e1)
        res["phase_ms"][tag] = {k: v / (a.iters + 1) for k, v in acc.items()}
        del tc, cc
        torch.cuda.empty_cache()
        if beta != 1:                                                     # same start, same number of iterations
            costs, _ = _fast.FusedNMF(X, U0, V0).run(a.check, 0.0, "mu", beta=beta)
            c_cc = cuda_core_steps(nmf.DeviceNMF(X, U0, V0, torch.float32), beta, a.check)
            res["objective"][tag] = {"iterations": a.check, "tensor_core": costs[-1], "cuda_core": c_cc,
                                     "rel_diff": abs(costs[-1] - c_cc) / abs(c_cc)}
            torch.cuda.empty_cache()
    y = res["median_it_per_s"]["beta=1"]["tensor_core"]
    res["speedup_over_cuda_core"] = {t: v["tensor_core"] / v["cuda_core"] for t, v in res["median_it_per_s"].items() if "cuda_core" in v}
    res["share_of_beta1_rate"] = {t: v["tensor_core"] / y for t, v in res["median_it_per_s"].items()}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_mu_beta.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
