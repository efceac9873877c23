"""Cost of precision "fp32x3" at C2 (65536 x 8192, rank 64): it/s of the 2-plane ("fp32") and the 3-plane ("fp32x3") tensor-core
path for HALS, MU beta = 1 and MU beta = 2, alternating in one process after warm-up, plus the time of each phase of an
iteration (CUDA events) and the card's name and power limit read in the same run.

    python tools/bench_fp32x3.py [--iters 20] [--reps 3] [--out DIR]

Prints one JSON document (and writes it to DIR/bench_fp32x3.json with --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nn-fac_b200"))
import torch  # noqa: E402

import nn_fac.config as config  # noqa: E402
from nn_fac import _fast  # noqa: E402

RULES = {"hals": ("hals", 2), "mu1": ("mu", 1), "mu2": ("mu", 2)}
PRECISIONS = ("fp32", "fp32x3")


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=65536)
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--r", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp32x3 needs a GPU")
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    m, n, r = a.m, a.n, a.r
    X = torch.rand((m, r), device=dev, generator=g) @ torch.rand((r, n), device=dev, generator=g)
    X += 0.1 * torch.rand((m, n), device=dev, generator=g)
    U0 = torch.rand((m, r), device=dev, generator=g)
    V0 = torch.rand((r, n), device=dev, generator=g)
    res = {"shape": [m, n, r], "iters_per_timing": a.iters, "card": card(), "it_per_s": {}, "phase_ms": {}}
    for tag, (rule, beta) in RULES.items():
        states = {}
        for prec in PRECISIONS:               # one resident state per precision, warmed up
            config.set_precision(prec)
            states[prec] = _fast.FusedNMF(X, U0, V0)
            states[prec].run(3, 0.0, rule, beta=beta)
        config.set_precision("auto")
        rates = {p: [] for p in PRECISIONS}
        for _ in range(a.reps):                # alternate the two paths
            for prec in PRECISIONS:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                states[prec].run(a.iters, 0.0, rule, beta=beta)
                torch.cuda.synchronize()
                rates[prec].append(a.iters / (time.perf_counter() - t0))
        res["it_per_s"][tag] = rates
        for prec in PRECISIONS:                # per-phase device times, in a run of their own
            st = states[prec]
            st.events = []
            st.run(a.iters, 0.0, rule, beta=beta)
            torch.cuda.synchronize()
            acc = {}
            for name, e0, e1 in st.events:
                acc[name] = acc.get(name, 0.0) + e0.elapsed_time(e1)
            st.events = None
            res["phase_ms"].setdefault(tag, {})[prec] = {k: v / (a.iters + 1) for k, v in acc.items()}
        del states
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_fp32x3.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
