#!/usr/bin/env python
"""Headline benchmark: NMF outer iterations / second, HALS and MU beta=1, 65536 x 8192, rank 64.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows M --cols N --rank R] [--dump-outputs DIR]

One "step" = one HALS outer iteration + one MU (beta=1) outer iteration (U update, V update, cost
each), every one on its own resident factor state.  `value` = 2K / T outer iterations per second
with X already resident in HBM; `e2e` is the same quantity through the public nn_fac.nmf.nmf()
call with host (pinned) arrays, upload and download inside the timed region.
Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement" for the roofline arithmetic.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "nn-fac_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "NMF outer iters/sec (HALS & MU beta=1) at 65536x8192 r=64"
UNIT = "outer_iters/s"
NOISE = 1.0   # X = W0 H0 + NOISE * mean(W0 H0) * E  ("spectrogram-like", residual ~ 10 %), SURVEY.md 8(d)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--m", "--rows", dest="m", type=int, default=65536)      # (--rows / --cols: torchrun's own parser chokes on --m)
    p.add_argument("--n", "--cols", dest="n", type=int, default=8192)
    p.add_argument("--rank", type=int, default=64)
    p.add_argument("--cpu-rows", type=int, default=16384, help="rows of the bounded CPU sample (all columns are kept)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-secondary", action="store_true", help="skip the secondary configs C1 / C4 / C5 / NTD-HALS (1 GPU)")
    p.add_argument("--c3", default="auto", choices=["auto", "on", "off"],
                   help="also run configs[2] (HALS rank 128 on 262144x32768, column-sharded); auto = when 8 GPUs are used")
    p.add_argument("--c3-m", type=int, default=262144)
    p.add_argument("--c3-n", type=int, default=32768)
    p.add_argument("--c3-rank", type=int, default=128)
    p.add_argument("--no-parity-n1", action="store_true", help="skip the sharded-vs-single-GPU self-check (N > 1)")
    p.add_argument("--c3-parity-full", action="store_true",
                   help="run the single-GPU self-check of C3 also when the matrix has more than 2^31 elements")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what they computed as DIR/<name>.npy: per rule (hals, mu) the factors U "
                        "(m x r) and V (r x n) and the costs of the timed iterations (see dump_outputs for the size cap)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


def ncu_traffic(phase):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel behind `phase`, from the committed
    `ncu --set full` capture of the last build at this shape (profiles/r2_ncu_full_final.json, else the mid-round
    profiles/r2_ncu_full_summaries.json: the first captured launch of that kernel instantiation is the C2 one); None when
    there is no capture of it."""
    kernels = {"hals.pass_U": ["tc_fused_kernel<0, 1, 0, 64>"], "hals.cross_V": ["tc_cross_kernel<64, 0>", "tc_cross_kernel<64>"],
               "mu.pass_U": ["tc_fused_kernel<1, 1, 1, 64>", "tc_fused_kernel<1, 1, 0, 64>"],
               "mu.pass_V": ["tc_fused_kernel<1, 0, 1, 64>", "tc_fused_kernel<1, 0, 0, 64>"]}.get(phase)
    path = next((q for q in (os.path.join(ROOT, "profiles", f) for f in ("r2_ncu_full_final.json", "r2_ncu_full_summaries.json"))
                 if os.path.exists(q)), None)
    if kernels is None or path is None:
        return None
    import re
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    blocks = [json.loads(blk) for blk in re.findall(r"\{.*?\n\}", open(path).read(), re.S)]
    for name in kernels:
        for d in blocks:
            if name in d.get("kernel", ""):
                tot = 0.0
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    val, u = d[key].split()
                    tot += float(val) * unit[u]
                return tot
    return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, flag in zip(names, r[5:9]):
                    if flag.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def synth_host(m, n, r, seed, dtype=np.float64):
    """Bounded-size synthetic problem for the CPU legs (same distribution as the device generator)."""
    rng = np.random.RandomState(seed)
    low = rng.rand(m, r) @ rng.rand(r, n)
    X = low + NOISE * low.mean() * rng.rand(m, n)
    return X.astype(dtype), rng.rand(m, r).astype(dtype), rng.rand(r, n).astype(dtype)


def _baseline_from(res, args, kind):
    """cpu_baseline object from the per-iteration seconds of a CPU run (scaled to the full shape, see oracle/ref_timing.py)."""
    value = 2.0 / (res["hals_s_per_iter"] + res["mu_s_per_iter"])
    rows = res["rows"]
    if rows == args.m:
        sample = f"full shape {args.m}x{args.n} r={args.rank} float64, {res['iters']} outer iteration(s) each of HALS and MU beta=1"
    else:
        sample = (f"{rows}x{args.n} r={args.rank} float64 row-subsample (all columns), {res['iters']} outer iteration(s) each of HALS and "
                  f"MU beta=1; the m-proportional part of an iteration is scaled by m/rows={res['scale']:g}, the V-side HALS solve "
                  f"(size independent of m, {res.get('hals_vsolve_s_per_iter', 0.0):.3f} s) is not")
    return {"value": value, "unit": UNIT, "cores": int(res.get("blas_threads") or os.cpu_count() or 1), "kind": kind, "sample": sample,
            "same_config": rows == args.m, "hals_its_per_s": 1.0 / res["hals_s_per_iter"], "mu_its_per_s": 1.0 / res["mu_s_per_iter"],
            "hals_sweeps_per_call": res.get("hals_sweeps_per_call"), "host_cpus": res.get("host_cpus"),
            "what": ("nn_fac.nmf.nmf(X64, r, init='custom', ..., deterministic=True) of the unmodified reference (oracle/_ref, tensorly "
                     "stand-in oracle/ref_shim)") if kind == "reference" else "numpy float64 port of the reference (oracle/nnfac_oracle.py)"}


def _port_timing(args, rows, iters):
    """Fallback when oracle/_ref is absent: the oracle port, same sampling and scaling as oracle/ref_timing.py."""
    from oracle import nnfac_oracle as orc
    from oracle.ref_timing import blas_threads
    X, U0, V0 = synth_host(rows, args.n, args.rank, seed=1)
    scale = args.m / rows
    orig, tv = orc.hals_nnls_acc, [0.0]

    def timed(UtM, *a, **kw):
        t0 = time.perf_counter()
        res = orig(UtM, *a, **kw)
        if UtM.shape[1] == args.n and rows != args.n:
            tv[0] += time.perf_counter() - t0
        return res
    orc.hals_nnls_acc = timed
    try:
        t0 = time.perf_counter()
        orc.compute_nmf(X, U0, V0, n_iter_max=iters, tol=0, update_rule="hals")
        t_hals = (time.perf_counter() - t0) / iters
    finally:
        orc.hals_nnls_acc = orig
    t0 = time.perf_counter()
    orc.compute_nmf(X, U0, V0, n_iter_max=iters, tol=0, update_rule="mu", beta=1)
    t_mu = (time.perf_counter() - t0) / iters
    v = tv[0] / iters
    return {"rows": rows, "scale": scale, "iters": iters, "hals_s_per_iter": (t_hals - v) * scale + v, "hals_vsolve_s_per_iter": v,
            "mu_s_per_iter": t_mu * scale, "blas_threads": blas_threads(), "host_cpus": os.cpu_count()}


def cpu_baseline(args, iters=1, in_process=False):
    """nn-fac's own CPU path on the host cores: the unmodified reference from oracle/_ref (kind "reference"), else the oracle
    port (kind "port").  Bounded sample: `--cpu-rows` rows of the m rows, all columns (see oracle/ref_timing.py for the scaling).
    The reference's package is called nn_fac like the product's, so from the GPU arm it runs in a subprocess."""
    rows = min(args.cpu_rows, args.m)
    have_ref = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "nn_fac"))
    if have_ref:
        try:
            if in_process:
                from oracle import ref_timing
                res = ref_timing.time_reference_nmf(args.m, args.n, args.rank, rows, iters, NOISE)
            else:
                cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_timing.py"), str(args.m), str(args.n), str(args.rank), str(rows),
                       str(iters), str(NOISE)]
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, check=True).stdout
                res = json.loads(out.strip().splitlines()[-1])
            res["iters"] = iters
            return _baseline_from(res, args, "reference")
        except Exception as e:                      # noqa: BLE001  (stated in the line, then the port is timed instead)
            note = f"reference run failed ({type(e).__name__}: {e}); "
    else:
        note = "oracle/_ref missing (python oracle/make_ref.py needs /root/reference); "
    base = _baseline_from(_port_timing(args, rows, iters), args, "port")
    base["sample"] = note + base["sample"]
    return base


def run_reference(args, rank):
    if rank != 0:
        return
    t0 = time.time()
    base = cpu_baseline(args, iters=max(1, min(args.steps, 3)), in_process=True)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 2000.0 / base["value"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"NMF {args.m}x{args.n} r={args.rank}: 1 HALS + 1 MU(beta=1) outer iteration per step",
                       "noise": NOISE, "note": "nn-fac's CPU path on the host cores (no GPU): " + base["what"] + "; " + base["sample"]},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t0}
    print(json.dumps(line))


def philox_problem(m, n, r, lo, hi, seed=20261018):
    """This rank's column block [lo, hi) of the synthetic problem (m x n, rank r): X = W0 H0 + NOISE * (r/4) * E with every
    entry a pure function of (seed, stream, global row, global column) (csrc/synth.cu), so any number of GPUs regenerates
    the same matrix shard by shard.  r/4 = E[W0 H0].  Returns device fp32 (X_p, U0, V0_p)."""
    import torch
    from nn_fac import _ops as ops
    W0 = ops.philox_uniform(m, r, seed=seed, stream_id=0)
    H0 = ops.philox_uniform(r, hi - lo, col0=lo, seed=seed, stream_id=1)
    X = torch.matmul(W0, H0)                       # data generation, not the timed path
    del W0, H0
    ops.philox_uniform(m, hi - lo, col0=lo, seed=seed, stream_id=2, scale=NOISE * r / 4.0, out=X, accumulate=True)
    U0 = ops.philox_uniform(m, r, seed=seed, stream_id=3)
    V0 = ops.philox_uniform(r, hi - lo, col0=lo, seed=seed, stream_id=4)
    return X, U0, V0


def run_c3(args, dev, world, rank, group, peak):
    """configs[2]: NMF HALS rank 128 on 262144 x 32768, column-sharded with the Gram / cross-product exchange on the U side
    (nmf.py:407-441, nnls.py:156-198).  Same timing rules as the headline; reports whole-job it/s and the per-GPU fraction of
    the 2 m n_p 4 + 4 (m + n_p) r 4 bytes per iteration and GPU of SURVEY.md 8(d)."""
    import torch
    import torch.distributed as dist
    from nn_fac import _fast
    from nn_fac.sharded import column_block
    m, n, r = args.c3_m, args.c3_n, args.c3_rank
    lo, hi = column_block(n, world, rank)
    torch.cuda.empty_cache()
    X, U0, V0 = philox_problem(m, n, r, lo, hi)
    st = _fast.FusedNMF(X, U0, V0, group=group)
    del X
    torch.cuda.empty_cache()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    st.run(args.warmup, 0.0, "hals")
    st.events, st.sweep_log = [], []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record()
    costs = st.run(args.steps, 0.0, "hals")[0]
    ev[1].record()
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    phases = {}
    for name, e0, e1 in st.events:
        phases.setdefault(name, []).append(e0.elapsed_time(e1))
    its = args.steps / (ms / 1e3)
    n_p = hi - lo
    bytes_gpu = 2 * m * n_p * 4 + 4 * (m + n_p) * r * 4
    out = {"config": f"C3: NMF HALS {m}x{n} r={r}, columns sharded over {world} GPU(s) ({n_p} columns each), fp32 storage",
           "outer_iters_per_s": its, "ms_per_iter": ms / args.steps, "n_gpus": world,
           "algorithmic_bytes_per_iter_per_gpu": bytes_gpu, "frac_of_hbm_roofline_per_gpu": bytes_gpu * its / 1e9 / peak,
           "phase_ms": {k: sum(v) / len(v) for k, v in phases.items()}, "final_cost": costs[-1],
           "hals_sweeps_per_call": [[float(v) for v in t.cpu().tolist()] for t in st.sweep_log[-3:]],
           "data": "synthetic, Philox keyed on (seed, global row, global column): identical for any number of GPUs"}
    sharded_sweeps = [[float(v) for v in t.cpu().tolist()] for t in st.sweep_log]
    del st
    torch.cuda.empty_cache()
    if world > 1 and not args.no_parity_n1 and (m * n <= 2 ** 31 or args.c3_parity_full):
        # self-check: rank 0 regenerates the WHOLE matrix from the same counters and repeats the run unsharded
        if rank == 0:
            X, U0, V0 = philox_problem(m, n, r, 0, n)
            one = _fast.FusedNMF(X, U0, V0)
            del X
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            c1 = one.run(args.warmup + args.steps, 0.0, "hals")[0]
            torch.cuda.synchronize()
            single_s = time.perf_counter() - t0
            single_sweeps = [[float(v) for v in t.cpu().tolist()] for t in one.sweep_log[-len(sharded_sweeps):]]
            out["parity_vs_n1"] = {"iterations": args.warmup + args.steps, "cost_single": c1[-1], "cost_sharded": costs[-1],
                                   "cost_rel_diff": abs(c1[-1] - costs[-1]) / abs(c1[-1]),
                                   "single_gpu_outer_iters_per_s": (args.warmup + args.steps) / single_s,
                                   "speedup_over_single_gpu": its / ((args.warmup + args.steps) / single_s),
                                   "sweeps_equal": single_sweeps == sharded_sweeps,
                                   "sweep_count_max_abs_diff": max((abs(a - b) for x, y in zip(single_sweeps, sharded_sweeps)
                                                                    for a, b in zip(x, y)), default=None)}
            del one
            torch.cuda.empty_cache()
        barrier()
    return out


def parity_vs_single_gpu(args, dev, world, rank, X_full, U0, V0_full, sharded_costs, sharded_sweeps):
    """Self-check of the sharded run (the driver's GPU tests are single-GPU): rank 0 repeats the SAME problem unsharded for the
    same number of iterations and compares objectives and HALS sweep counts."""
    import torch
    from nn_fac import _fast
    if rank != 0:
        return None
    iters = args.warmup + args.steps
    out = {"iterations": iters, "shape": list(X_full.shape), "rank": int(U0.shape[1])}
    for rule in ("hals", "mu"):
        st = _fast.FusedNMF(X_full, U0, V0_full)
        costs = st.run(iters, 0.0, rule)[0]
        out[f"{rule}_cost_single"] = costs[-1]
        out[f"{rule}_cost_sharded"] = sharded_costs[rule]
        out[f"{rule}_cost_rel_diff"] = abs(costs[-1] - sharded_costs[rule]) / abs(costs[-1])
        if rule == "hals":
            single = [[float(v) for v in t.cpu().tolist()] for t in st.sweep_log[-len(sharded_sweeps):]] if sharded_sweeps else []
            out["hals_sweeps_single_last"] = single
            out["hals_sweeps_sharded_last"] = sharded_sweeps
            out["hals_sweeps_equal"] = single == sharded_sweeps
            out["hals_sweep_count_max_abs_diff"] = max((abs(a - b) for x, y in zip(single, sharded_sweeps) for a, b in zip(x, y)),
                                                       default=None)
        del st
        torch.cuda.empty_cache()
    return out


DUMP_BYTES = 63 * 10 ** 6      # array data of --dump-outputs: with the .npy headers, the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes every array of `arrays` (name -> float32 / float64 numpy array) as out_dir/<name>.npy.  If they add up to more
    than DUMP_BYTES, every matrix keeps the same fraction of its longer axis (rows of U, columns of V), chosen by a fixed seed,
    so that two runs with the same arguments write the same entries."""
    os.makedirs(out_dir, exist_ok=True)
    mats = sum(a.nbytes for a in arrays.values() if a.ndim == 2)
    rest = sum(a.nbytes for a in arrays.values() if a.ndim != 2)
    keep = min(1.0, (DUMP_BYTES - rest) / mats) if mats else 1.0
    for name, a in arrays.items():
        if keep < 1.0 and a.ndim == 2:
            axis = 0 if a.shape[0] >= a.shape[1] else 1
            idx = np.sort(np.random.RandomState(0).choice(a.shape[axis], max(1, int(a.shape[axis] * keep)), replace=False))
            a = np.take(a, idx, axis=axis)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def timed_outputs(states, costs, fused, world):
    """What a caller of the timed path receives for each rule: U (m x r), V (r x n) and the costs of the timed iterations.
    Column-sharded runs gather the column blocks of V (every rank must call this)."""
    import torch.distributed as dist
    out = {}
    for rule, st in states.items():
        U, V = st.factors() if fused else (st.U, st.V)
        V = V.cpu().numpy()
        if world > 1:
            blocks = [None] * world
            dist.all_gather_object(blocks, V)
            V = np.concatenate(blocks, axis=1)
        out[f"{rule}_U"], out[f"{rule}_V"] = U.cpu().numpy(), V
        out[f"{rule}_costs"] = np.asarray(costs[rule], dtype=np.float64)
    return out


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import nn_fac.nmf as nmf
    from nn_fac import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m, n, r = args.m, args.n, args.rank

    # ---- synthetic data, generated on the device (not part of the timed path) ----
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    W0 = torch.rand((m, r), generator=gen, device=dev)
    H0 = torch.rand((r, n), generator=gen, device=dev)
    X = W0 @ H0
    X.add_(torch.rand((m, n), generator=gen, device=dev), alpha=NOISE * float(X.mean()))
    U0 = torch.rand((m, r), generator=gen, device=dev)
    V0 = torch.rand((r, n), generator=gen, device=dev)
    del W0, H0
    sp, fixed, norm = [None, None], [], [False, False]

    from nn_fac import _fast
    from nn_fac.sharded import column_block
    fused = args.rank <= 64
    group = None
    X_full = V0_full = None
    if world > 1:
        # every rank generated the same X (same seed, same generator); it keeps its own column block only
        assert fused, "the sharded headline covers rank <= 64 (MU beta = 1)"
        lo, hi = column_block(n, world, rank)
        if rank == 0 and not args.no_parity_n1:
            X_full, V0_full = X, V0
        X, V0 = X[:, lo:hi].contiguous(), V0[:, lo:hi].contiguous()
        group = dist.group.WORLD
        torch.cuda.empty_cache()
    if fused:
        states = {"hals": _fast.FusedNMF(X, U0, V0, group=group), "mu": _fast.FusedNMF(X, U0, V0, group=group)}
    else:
        states = {"hals": nmf.DeviceNMF(X, U0, V0, torch.float32), "mu": nmf.DeviceNMF(X, U0, V0, torch.float32)}

    def run_rule(rule, iters):
        """`iters` outer iterations of one rule on its resident state; returns the list of costs."""
        st = states[rule]
        if fused:
            return st.run(iters, 0.0, rule, sp, fixed, norm)[0]
        return [st.step(rule, 2 if rule == "hals" else 1, sp, fixed, norm) for _ in range(iters)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.warmup > 0:
        run_rule("hals", args.warmup)
        run_rule("mu", args.warmup)
    # phase timers (CUDA events on the launching stream) are collected during the timed region
    for s in states.values():
        s.events = []
        if fused:
            s.sweep_log = []
    launches0 = _lib.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    barrier()
    with ClockSampler(local_rank) as clocks:
        ev[0].record()
        c1 = run_rule("hals", args.steps)
        ev[1].record()
        c2 = run_rule("mu", args.steps)
        ev[2].record()
        barrier()
    costs = (c1[-1], c2[-1])
    total_ms = ev[0].elapsed_time(ev[2])
    t_rule = {"hals": ev[0].elapsed_time(ev[1]), "mu": ev[1].elapsed_time(ev[2])}
    launches = _lib.launch_count() - launches0
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = 2.0 * args.steps / (total_ms / 1e3)
    if args.dump_outputs:
        outputs = timed_outputs(states, {"hals": c1, "mu": c2}, fused, world)
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)

    # ---- per-phase breakdown and roofline of the dominant kernel ----
    phases = {}
    for rule, s in states.items():
        for name, e0, e1 in s.events:
            phases.setdefault(f"{rule}.{name}", []).append(e0.elapsed_time(e1))
    phase_ms = {k: sum(v) / len(v) for k, v in phases.items()}
    peak, peak_src = measured_peaks()
    n_loc = X.shape[1]
    x_bytes = m * n_loc * 4                              # this rank's block of X
    dom = max((k for k in phase_ms if "cross" in k or "update" in k or "pass" in k), key=lambda k: phase_ms[k], default=None)
    roofline = None
    if dom is not None:
        fac_bytes = 2 * (m + n_loc) * r * 4
        algo = x_bytes + fac_bytes                      # one pass over X + both factor-sized operands in/out
        ach = algo / (phase_ms[dom] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_traffic(dom) if (m, n, r, world) == (65536, 8192, 64, 1) else None,
                    "traffic_source": "ncu --set full capture of this kernel at this shape (profiles/r2_ncu_full_final.json)",
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": algo,
                    "ms_per_launch": phase_ms[dom]}
    algo_iter = 2 * m * n * 4 + 4 * (m + n) * r * 4     # SURVEY.md 8(d): bytes per outer iteration (whole job)
    per_rule = {k: args.steps / (t_rule[k] / 1e3) for k in t_rule}
    iter_roofline = {k: algo_iter * per_rule[k] / 1e9 / (peak * world) for k in per_rule}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"NMF {m}x{n} r={r}: 1 HALS + 1 MU(beta=1) outer iteration per step",
                       "noise": NOISE, "l2": f"X block per GPU ({x_bytes / 1e9:.2f} GB) larger than L2 (126 MB); no flush needed", "parallelism": f"cols/{world}"},
            "hals_its_per_s": per_rule["hals"], "mu_its_per_s": per_rule["mu"],
            "frac_of_hbm_roofline_per_iteration": iter_roofline,
            "phase_ms": phase_ms, "final_costs": {"hals": costs[0], "mu": costs[1]},
            "hals_sweeps_per_call": ([[float(v) for v in t.cpu().tolist()] for t in states["hals"].sweep_log[-3:]] if fused
                                     else [float(x) for x in states["hals"].hals_stats[:, 3].cpu().tolist()]),
            "gpu_launches": int(launches), "roofline": roofline}

    if rank == 0:
        line["clocks"] = clocks.summary()
    if world > 1 and not args.no_parity_n1:
        sharded_sweeps = [[float(v) for v in t.cpu().tolist()] for t in states["hals"].sweep_log[-3:]] if fused else []
        chk = parity_vs_single_gpu(args, dev, world, rank, X_full, U0, V0_full, {"hals": costs[0], "mu": costs[1]}, sharded_sweeps)
        del X_full, V0_full
        barrier()
        if rank == 0:
            line["parity_vs_n1"] = chk

    # ---- end to end through the public API with host buffers ----
    if not args.no_e2e:
        from nn_fac.sharded import compute_nmf_sharded
        n_loc = X.shape[1]
        Xh = torch.empty((m, n_loc), dtype=torch.float32, pin_memory=True); Xh.copy_(X)
        Uh = torch.empty((m, r), dtype=torch.float32, pin_memory=True); Uh.copy_(U0)
        Vh = torch.empty((r, n_loc), dtype=torch.float32, pin_memory=True); Vh.copy_(V0)
        del states, s, X, U0, V0
        torch.cuda.empty_cache()
        k = args.steps

        def call(rule, beta, iters):
            if world == 1:
                return nmf.nmf(Xh.numpy(), r, init="custom", U_0=Uh.numpy(), V_0=Vh.numpy(), n_iter_max=iters, tol=0,
                               update_rule=rule, beta=beta, return_costs=True, deterministic=True)
            return compute_nmf_sharded(Xh.numpy(), r, Uh.numpy(), Vh.numpy(), n_iter_max=iters, tol=0,
                                       update_rule=rule, beta=beta, return_costs=True, group=group)

        call("hals", 2, 1)      # untimed warm-up of the public path (allocator blocks, pinned-copy path)
        call("mu", 1, 1)
        t_e2e = 0.0
        for rule, beta in (("hals", 2), ("mu", 1)):
            barrier()
            t0 = time.perf_counter()
            U, V, cs, _ = call(rule, beta, k)
            barrier()
            t_e2e += time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_e2e = float(t.item())
        h2d = 2 * (m * n_loc * 4 + (m + n_loc) * r * 4) / k     # per rank
        d2h = 2 * ((m + n_loc) * r * 4) / k + 2 * 8
        api = "nn_fac.nmf.nmf" if world == 1 else "nn_fac.sharded.compute_nmf_sharded"
        line["e2e"] = {"value": 2.0 * k / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "note": f"{api}(pinned host arrays, n_iter_max={k}) once per rule: X uploaded once per call, "
                               "bytes (per rank) amortised over the call's iterations; one untimed 1-iteration call per rule first; "
                               "wall clock, max over ranks"}
    run_c3_now = args.c3 == "on" or (args.c3 == "auto" and world == 8)
    if run_c3_now:
        try:
            states = s = X = U0 = V0 = None            # noqa: F841  (free the headline's state before the 4.3 GB blocks of C3)
            torch.cuda.empty_cache()
            line["c3"] = run_c3(args, dev, world, rank, group, peak)
        except Exception as e:                        # noqa: BLE001
            line["c3"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0 and world == 1 and not args.no_secondary:
        states = s = X = U0 = V0 = None                # noqa: F841
        torch.cuda.empty_cache()
        from tools import secondary
        line["secondary"] = secondary.all_secondary(peak_gbs=peak, iters=10)
        line["secondary"]["note"] = ("BASELINE.json configs[0], [3], [4] and the reference's default NTD rule on this GPU, run after "
                                     "the headline (outside its timed region); CUDA events except c1 (wall clock of the public call)")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args, iters=1)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
